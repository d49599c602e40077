"""The split-M weight-gradient reductions on their own against fp64, with every row live up to the last.

Inside a learner step the last rows of these reductions are zero or masked (the online Q of t = TT - 1 is never part of
the loss; the last episodes are usually shorter than the window), so a kernel that dropped or misread a chunk's tail would
pass the learner tests.  Here dY ~ N(0, 1) on every row and each raw per-chunk partial is checked against its own rows:
  * assert_close(.., 1e-5), the project's norm-wise bar;
  * element-wise |err| <= 1e-5 * sum_m |dY[m, n] A[m, k]|, and exactly 0 where that sum is 0;
  * the reference recomputed WITHOUT the last row of the chunk must fail one of those bars (the data makes the tail
    visible).
Operands sit inside NaN-filled buffers (rows past M, columns past Nout / K inside ldy / lda, the `shift` rows before A);
partial buffers start as NaN with a NaN tail that must survive.

Long single chunks on the fp32 FFMA kernel are not run past 65 537 rows: one thread sums its chunk in one sequential
fp32 chain, whose norm-wise error grows like ~0.3 u sqrt(n) (u = 2^-24): a numpy emulation of such a chain gives 8.7e-6
norm-wise and 1.7e-5 max at n = 200 000 rows, so a correct kernel would exceed the 1e-5 bar there.  The learner's
chunking never hands that kernel such chunks.
"""
import ctypes as C

import numpy as np
import pytest
import torch as th

from ma_league_b200 import _native as nat
from tests.helpers import RTOL, assert_close, max_err, rel_err
from tests.reduce_ref import F64, agent_rows, chunk_sums, dense_rows, fc2_sums, gru_sums, n_chunks, state_rows

pytestmark = pytest.mark.gpu
DEV = "cuda"
NAN = float("nan")
TAIL = 67                                   # NaN floats behind every partial buffer
FLAVOURS = [nat.RED_FFMA, nat.RED_TC_MN0, nat.RED_TC_MN1, nat.RED_TC_MN2, nat.RED_TC3]
FNAME = {nat.RED_FFMA: "ffma", nat.RED_TC_MN0: "tc_mn0", nat.RED_TC_MN1: "tc_mn1", nat.RED_TC_MN2: "tc_mn2",
         nat.RED_TC3: "tc3"}
FFMA_MAX_CHUNK = 65537                      # see the module docstring


def gen(seed):
    return th.Generator(device=DEV).manual_seed(seed)


def buffer2d(rows, cols, ld, off, g, before=0, valid=None):
    """[rows, cols] view (row stride ld) at float offset off + before*ld of a NaN-filled store; rows < valid get N(0, 1)."""
    store = th.full(((before + rows + 2) * ld + off + 8,), NAN, device=DEV)
    start = off + before * ld
    view = store[start:start + rows * ld].view(rows, ld)[:, :cols]
    v = rows if valid is None else valid
    if v > 0:
        view[:v] = th.randn(v, cols, generator=g, device=DEV)
    return store, view, store.data_ptr() + 4 * start


def partial_buffer(n):
    return th.full((n + TAIL,), NAN, device=DEV)


def take_partial(buf, shape, what):
    n = int(np.prod(shape))
    assert bool(th.isnan(buf[n:]).all()), "%s: the NaN tail behind the partials was written" % what
    out = buf[:n].view(*shape)
    assert bool(th.isfinite(out).all()), "%s: a partial was not written or is not finite" % what
    return out


def check_chunks(what, W, B, ref):
    """Per-chunk bars on the kernel's partials W [nc, ...] / B [nc, ...] (B may be None) against a chunk_sums dict."""
    r = {k: v.cpu().numpy() for k, v in ref.items()}
    W = W.double().cpu().numpy()
    B = B.double().cpu().numpy() if B is not None else None
    worst, live, visible = 0.0, 0, 0
    for c in range(W.shape[0]):
        pairs = [("W", W[c])] + ([("B", B[c])] if B is not None else [])
        tail_passes = True
        contributes = False
        for key, got in pairs:
            ref_c, ab, drop = r[key][c], r[key + "_abs"][c], r[key + "_drop"][c]
            assert_close(got, ref_c, RTOL, "%s chunk %d d%s" % (what, c, key))
            err = np.abs(got - ref_c)
            bad = err > RTOL * ab
            assert not bad.any(), "%s chunk %d d%s: %d entries over 1e-5 * sum|dY A| (first %s: %r vs %r, scale %r)" % (
                what, c, key, int(bad.sum()), np.argwhere(bad)[0], got[bad][0], ref_c[bad][0], ab[bad][0])
            nz = ab > 0
            if nz.any():
                worst = max(worst, float((err[nz] / ab[nz]).max()))
            contributes = contributes or not np.array_equal(ref_c, drop)
            if not (rel_err(got, drop) <= RTOL and max_err(got, drop) <= RTOL and (np.abs(got - drop) <= RTOL * ab).all()):
                tail_passes = False
        if contributes:
            live += 1
            visible += not tail_passes
    assert live > 0, "%s: no chunk has a live last row" % what
    assert visible == live, "%s: without its last row, %d of %d chunks still pass every bar" % (what, live - visible, live)
    print("%s: %d chunks, worst |err| / sum|dY A| = %.2e" % (what, W.shape[0], worst))
    return worst


def stat_key(flavour, probs):
    if flavour == nat.RED_FFMA:
        return "reduce_ffma"
    return "reduce_tc_swap" if all(p["Nout"] <= 64 < p["K"] for p in probs) else "reduce_tc"


def run_generic(flavour, a_kind, probs, batch=None, agent_input=0):
    """probs: dicts with M, rpc, K, Nout, shift, dY (view), dY_ptr, A_ptr / lda (dense), bias (bool).
    Launches mal_debug_reduce, checks the sentinels and the flavour counter; returns [(W, B)] per problem."""
    arr = (nat.RedProb * len(probs))()
    bufs = []
    for i, p in enumerate(probs):
        nc = n_chunks(p["M"], p["rpc"])
        wb = partial_buffer(nc * p["Nout"] * p["K"])
        bb = partial_buffer(nc * p["Nout"]) if p.get("bias", True) else None
        bufs.append((nc, wb, bb))
        arr[i] = nat.RedProb(p["M"], p["rpc"], p["K"], p["Nout"], p.get("shift", 0), p["dY_ptr"], p["dY"].stride(0),
                             p.get("A_ptr", 0) or None, p.get("lda", 0), wb.data_ptr(), bb.data_ptr() if bb is not None else None)
    key = stat_key(flavour, probs)
    before = nat.lib().mal_stat(key.encode())
    nat.check(nat.lib().mal_debug_reduce(flavour, a_kind, len(probs), arr, C.byref(batch) if batch is not None else None,
                                         agent_input, nat.current_stream()), "mal_debug_reduce")
    th.cuda.synchronize()
    assert nat.lib().mal_stat(key.encode()) == before + 1, "flavour %s did not run %s" % (FNAME[flavour], key)
    out = []
    for p, (nc, wb, bb) in zip(probs, bufs):
        W = take_partial(wb, (nc, p["Nout"], p["K"]), "part_w")
        B = take_partial(bb, (nc, p["Nout"]), "part_b") if bb is not None else None
        out.append((W, B))
    return out


def dense_prob(M, Nout, K, rpc, shift, vec, g, bias=True):
    """dY [M, Nout] and A [M - shift, K] in NaN-padded buffers: vec = aligned rows (ld % 4 == 0, 16-byte pointers),
    otherwise ld % 4 != 0 and pointers one float off."""
    off = 0 if vec else 1
    ldy = (Nout + 3) // 4 * 4 + 4 if vec else Nout + 3
    lda = (K + 3) // 4 * 4 + 4 if vec else K + 1 + (K % 2)
    ys, y, yp = buffer2d(M, Nout, ldy, off, g)
    na = max(M - shift, 0)
    as_, a, ap = buffer2d(na, K, lda, off, g, before=shift)
    return dict(M=M, rpc=rpc, K=K, Nout=Nout, shift=shift, dY=y, dY_ptr=yp, A_ptr=ap, lda=lda, bias=bias,
                keep=(ys, as_), A=a)


def dy_rows(y):
    return lambda m0, m1: y[m0:m1].to(F64)


# ---------------------------------------------------------------------------------------------------------------------
# batches for the state / agent-input loaders (NaN wherever no row < M may read)
# ---------------------------------------------------------------------------------------------------------------------
def state_batch(B, T, S, M, K, shift, vec, g):
    TT = T + 1
    ld = S if vec and S % 4 == 0 else S + (1 if S % 2 == 0 else 2)
    off = 0 if vec else 1
    store = th.full((B * TT * ld + off + 8,), NAN, device=DEV)
    state = store[off:off + B * TT * ld].view(B, TT, ld)[:, :, :S]
    vals = th.randn(B * T, K, generator=g, device=DEV)
    vals[M:] = NAN
    state[:, shift:shift + T, :K] = vals.view(B, T, K)
    b = nat.Batch(B, TT, 1, 1, 1, S)
    b.state = nat.Field(store.data_ptr() + 4 * off, TT * ld, ld)
    return b, state, store


def agent_batch(B, TT, N, A, OBS, flags, M, vec, g):
    R = B * N
    ldo = N * OBS if vec and (N * OBS) % 4 == 0 else N * OBS + (1 if (N * OBS) % 2 == 0 else 2)
    off = 0 if vec else 1
    ostore = th.full((B * TT * ldo + off + 8,), NAN, device=DEV)
    obs = ostore[off:off + B * TT * ldo].view(B, TT, ldo)[:, :, :N * OBS].view(B, TT, N, OBS)
    ldh = N * A + 3
    hstore = th.full((B * TT * ldh + 8,), NAN, device=DEV)
    onehot = hstore[:B * TT * ldh].view(B, TT, ldh)[:, :, :N * A].view(B, TT, N, A)
    m = th.arange(TT * R, device=DEV)
    t, rr = m // R, m % R
    b_, n_ = rr // N, rr % N
    live = m < M
    obs[b_[live], t[live], n_[live]] = th.randn(int(live.sum()), OBS, generator=g, device=DEV)
    read = (m + R < M) & (t < TT - 1)                        # onehot[b, t, n] is read by row (t + 1) R + b N + n
    onehot[b_[read], t[read], n_[read]] = th.randn(int(read.sum()), A, generator=g, device=DEV)
    bs = nat.Batch(B, TT, N, A, OBS, 1)
    bs.obs = nat.Field(ostore.data_ptr() + 4 * off, TT * ldo, ldo)
    bs.onehot = nat.Field(hstore.data_ptr(), TT * ldh, ldh)
    last, aid = not (flags & nat.IN_NO_LAST_ACTION), not (flags & nat.IN_NO_AGENT_ID)
    d_in = OBS + (A if last else 0) + (N if aid else 0)
    return bs, agent_rows(obs, onehot, last, aid), d_in, (ostore, hstore)


# ---------------------------------------------------------------------------------------------------------------------
# generic reductions (k_reduce_group, k_reduce_tc<.., 0 | 1 | 2>, k_reduce_tc3)
# ---------------------------------------------------------------------------------------------------------------------
DENSE_SHAPES = [(192, 64), (128, 64), (64, 64), (64, 214), (64, 246), (64, 256), (320, 64), (192, 80), (1, 3), (64, 59)]


@pytest.mark.parametrize("vec", [True, False], ids=["vec", "scalar"])
@pytest.mark.parametrize("shift", [0, 7])
@pytest.mark.parametrize("Nout,K", DENSE_SHAPES)
@pytest.mark.parametrize("flavour", FLAVOURS, ids=[FNAME[f] for f in FLAVOURS])
def test_dense_shapes(flavour, Nout, K, shift, vec):
    for M, rpc in ((257, 64), (1000, 576)):
        g = gen(M + Nout * 7 + K * 13 + shift)
        p = dense_prob(M, Nout, K, rpc, shift, vec, g)
        (W, B), = run_generic(flavour, nat.RED_A_DENSE, [p])
        ref = chunk_sums(dy_rows(p["dY"]), dense_rows(p["A"], shift), M, rpc)
        check_chunks("dense %s M=%d rpc=%d %dx%d shift=%d %s" % (FNAME[flavour], M, rpc, Nout, K, shift,
                                                                "vec" if vec else "scalar"), W, B, ref)


SWEEP_M = [1, 31, 32, 33, 255, 257, 65537, 200003]


def sweep_rpcs(flavour, M):
    big = M if flavour != nat.RED_FFMA or M <= FFMA_MAX_CHUNK else 16384
    return [(64, True), (320, False), (576, True), ((big + 63) // 64 * 64 + (64 if M % 2 else 0), False)]


@pytest.mark.parametrize("M", SWEEP_M)
@pytest.mark.parametrize("loader", ["dense", "dense_shift", "state", "agent"])
@pytest.mark.parametrize("flavour", FLAVOURS, ids=[FNAME[f] for f in FLAVOURS])
def test_row_sweep(flavour, loader, M):
    for rpc, vec in sweep_rpcs(flavour, M):
        g = gen(M * 3 + rpc)
        what = "%s %s M=%d rpc=%d %s" % (loader, FNAME[flavour], M, rpc, "vec" if vec else "scalar")
        if loader.startswith("dense"):
            shift = 15 if loader == "dense_shift" else 0
            p = dense_prob(M, 128, 80, rpc, shift, vec, g)
            (W, B), = run_generic(flavour, nat.RED_A_DENSE, [p])
            ref = chunk_sums(dy_rows(p["dY"]), dense_rows(p["A"], shift), M, rpc)
        elif loader == "state":
            T, S, K, Nout = 7, 84 if vec else 82, 80, 160
            Bn = (M + T - 1) // T
            bs, state, keep = state_batch(Bn, T, S, M, K, 0, vec, g)
            ys, y, yp = buffer2d(M, Nout, Nout + (0 if vec else 3), 0 if vec else 1, g)
            (W, B), = run_generic(flavour, nat.RED_A_STATE, [dict(M=M, rpc=rpc, K=K, Nout=Nout, dY=y, dY_ptr=yp)], bs)
            ref = chunk_sums(dy_rows(y), state_rows(state, T, K), M, rpc)
        else:
            N, A, OBS, Bn = 5, 11, 52 if vec else 47, 3                     # R = 15 < 16; d_in = 68 (47: 63)
            R = Bn * N
            TT = max(2, (M + R - 1) // R + 1)
            bs, rows, d_in, keep = agent_batch(Bn, TT, N, A, OBS, 0, M, vec, g)
            ys, y, yp = buffer2d(M, 64, 64 if vec else 67, 0 if vec else 1, g)
            (W, B), = run_generic(flavour, nat.RED_A_AGENT_IN, [dict(M=M, rpc=rpc, K=d_in, Nout=64, dY=y, dY_ptr=yp)], bs, 0)
            ref = chunk_sums(dy_rows(y), rows, M, rpc)
        check_chunks(what, W, B, ref)


@pytest.mark.parametrize("vec", [True, False], ids=["vec", "scalar"])
@pytest.mark.parametrize("Nout,K,S", [(160, 80, 80), (32, 80, 80), (192, 80, 83), (1, 3, 5), (64, 59, 64), (96, 36, 38)])
@pytest.mark.parametrize("flavour", FLAVOURS, ids=[FNAME[f] for f in FLAVOURS])
def test_state_shapes(flavour, Nout, K, S, vec):
    for M, rpc, T, shift in ((257, 64, 9, 0), (1000, 320, 13, 1)):
        g = gen(Nout + K + S + M)
        Bn = (M + T - 1) // T + 1
        bs, state, keep = state_batch(Bn, T, S, M, K, shift, vec, g)
        ys, y, yp = buffer2d(M, Nout, Nout + (4 if vec else 1), 0 if vec else 1, g)
        (W, B), = run_generic(flavour, nat.RED_A_STATE, [dict(M=M, rpc=rpc, K=K, Nout=Nout, shift=shift, dY=y, dY_ptr=yp)], bs)
        check_chunks("state %s M=%d rpc=%d %dx%d S=%d shift=%d %s" % (FNAME[flavour], M, rpc, Nout, K, S, shift,
                                                                     "vec" if vec else "scalar"),
                     W, B, chunk_sums(dy_rows(y), state_rows(state, T, K, shift), M, rpc))


AGENT_CASES = [   # (N, A, OBS, B, flags): d_in below / at / just over 128, 214, 256; R < 16; OBS % 4 != 0; N = 1, 16, 17, 20
    (5, 11, 48, 3, 0), (16, 12, 100, 2, 0), (17, 11, 101, 1, 0), (20, 26, 168, 4, 0), (1, 3, 256, 5, 3),
    (1, 3, 60, 7, 0), (20, 26, 90, 2, nat.IN_NO_LAST_ACTION), (20, 26, 90, 2, nat.IN_NO_AGENT_ID), (5, 11, 45, 3, 3),
]


@pytest.mark.parametrize("vec", [True, False], ids=["vec", "scalar"])
@pytest.mark.parametrize("N,A,OBS,Bn,flags", AGENT_CASES)
@pytest.mark.parametrize("flavour", FLAVOURS, ids=[FNAME[f] for f in FLAVOURS])
def test_agent_input_shapes(flavour, N, A, OBS, Bn, flags, vec):
    R = Bn * N
    TT = (700 + R - 1) // R + 1
    for M, rpc in ((TT * R, 320), (TT * R - 7, 64)):
        g = gen(N * 100 + OBS + M)
        bs, rows, d_in, keep = agent_batch(Bn, TT, N, A, OBS, flags, M, vec, g)
        ys, y, yp = buffer2d(M, 64, 64 if vec else 65, 0 if vec else 1, g)
        (W, B), = run_generic(flavour, nat.RED_A_AGENT_IN, [dict(M=M, rpc=rpc, K=d_in, Nout=64, dY=y, dY_ptr=yp)], bs, flags)
        check_chunks("agent %s M=%d rpc=%d N=%d OBS=%d d_in=%d flags=%d %s" % (FNAME[flavour], M, rpc, N, OBS, d_in, flags,
                                                                             "vec" if vec else "scalar"),
                     W, B, chunk_sums(dy_rows(y), rows, M, rpc))


@pytest.mark.parametrize("flavour", FLAVOURS, ids=[FNAME[f] for f in FLAVOURS])
def test_groups(flavour):
    """Three problems per launch, as the learner groups them: the tile -> problem lookup, problems with different chunk
    counts (the early exit of the surplus chunks), and the swap decision (swapped only when every problem is swap-shaped)."""
    # the GRU weight gradients as the unfused path launches them: W_ih | W_hh (r, z) | W_hh (n) out of one d_g buffer
    R, TT = 96, 7
    M = R * TT
    for rpc in (128, 320):
        g = gen(rpc)
        gs, d_g, gp = buffer2d(M, 256, 256, 0, g)
        xs, x, xp = buffer2d(M, 64, 64, 0, g)
        hs, h, hp = buffer2d(M - R, 64, 64, 0, g, before=R)
        probs = [dict(M=M, rpc=rpc, K=64, Nout=192, dY=d_g, dY_ptr=gp, A_ptr=xp, lda=64),
                 dict(M=M, rpc=rpc, K=64, Nout=128, shift=R, dY=d_g, dY_ptr=gp, A_ptr=hp, lda=64),
                 dict(M=M, rpc=rpc, K=64, Nout=64, shift=R, dY=d_g, dY_ptr=gp + 4 * 192, A_ptr=hp, lda=64)]
        out = run_generic(flavour, nat.RED_A_DENSE, probs)
        for (W, B), (lo, hi, a, s), name in zip(out, ((0, 192, x, 0), (0, 128, h, R), (192, 256, h, R)), ("W_ih", "W_hh_rz", "W_hh_n")):
            ref = chunk_sums(lambda m0, m1: d_g[m0:m1, lo:hi].to(F64), dense_rows(a, s), M, rpc)
            check_chunks("group gru %s %s rpc=%d" % (FNAME[flavour], name, rpc), W, B, ref)
    # mixer-like state problems with different chunk counts (16, 4 and 2 chunks); one is swap-shaped, the group is not
    T, S, M = 9, 80, 1000
    g = gen(5)
    bs, state, keep = state_batch((M + T - 1) // T, T, S, M, S, 0, True, g)
    probs = []
    for Nout, rpc, vec in ((160, 64, True), (32, 320, False), (192, 576, True)):
        ys, y, yp = buffer2d(M, Nout, Nout + (0 if vec else 3), 0 if vec else 1, g)
        probs.append(dict(M=M, rpc=rpc, K=S, Nout=Nout, dY=y, dY_ptr=yp, keep=ys))
    for (W, B), p in zip(run_generic(flavour, nat.RED_A_STATE, probs, bs), probs):
        check_chunks("group state %s %dx%d rpc=%d" % (FNAME[flavour], p["Nout"], S, p["rpc"]), W, B,
                     chunk_sums(dy_rows(p["dY"]), state_rows(state, T, S), M, p["rpc"]))
    # swap-shaped dense problems (Nout <= 64 < K) with different row counts and chunkings; the last has no bias
    probs = [dense_prob(700, 64, 214, 64, 0, True, g), dense_prob(513, 64, 246, 320, 3, False, g),
             dense_prob(97, 1, 256, 576, 0, True, g, bias=False)]
    for (W, B), p in zip(run_generic(flavour, nat.RED_A_DENSE, probs), probs):
        check_chunks("group swap %s %dx%d M=%d rpc=%d" % (FNAME[flavour], p["Nout"], p["K"], p["M"], p["rpc"]), W, B,
                     chunk_sums(dy_rows(p["dY"]), dense_rows(p["A"], p["shift"]), p["M"], p["rpc"]))


# ---------------------------------------------------------------------------------------------------------------------
# k_reduce_gru
# ---------------------------------------------------------------------------------------------------------------------
def run_gru(M1, R, rpc, g):
    xs, x, xp = buffer2d(M1, 64, 64, 0, g)
    hs, h, hp = buffer2d(M1, 64, 64, 0, g, before=R)                   # the R rows before hout must never be read
    gs, d_g, gp = buffer2d(M1, 256, 256, 0, g)
    nc = n_chunks(M1, rpc)
    bufs = [partial_buffer(nc * n) for n in (192 * 64, 192, 128 * 64, 128, 64 * 64, 64)]
    before = nat.lib().mal_stat(b"reduce_tc")
    nat.check(nat.lib().mal_debug_reduce_gru(xp, hp, gp, M1, R, rpc, *[b.data_ptr() for b in bufs], nat.current_stream()),
              "mal_debug_reduce_gru")
    th.cuda.synchronize()
    assert nat.lib().mal_stat(b"reduce_tc") == before + 1
    shapes = [(nc, 192, 64), (nc, 192), (nc, 128, 64), (nc, 128), (nc, 64, 64), (nc, 64)]
    parts = [take_partial(b, s, "k_reduce_gru partial") for b, s in zip(bufs, shapes)]
    return parts, gru_sums(x, h, d_g, R, rpc)


@pytest.mark.parametrize("TT", [1, 2, 201])
@pytest.mark.parametrize("R", [1, 5, 15, 16, 17, 96, 320])
def test_reduce_gru(R, TT):
    M1 = TT * R
    for rpc in sorted({64, 320, (M1 + 63) // 64 * 64}):
        parts, refs = run_gru(M1, R, rpc, gen(R * 1000 + TT + rpc))
        for i, name in enumerate(("W_ih", "W_hh_rz", "W_hh_n")):
            W, B = parts[2 * i], parts[2 * i + 1]
            if name != "W_ih":   # a chunk inside the first R rows pairs with h_{-1} = 0: its W_hh partials are exactly 0
                for c in range(W.shape[0]):
                    if (c + 1) * rpc <= R:
                        assert bool((W[c] == 0).all()), "k_reduce_gru R=%d chunk %d: W_hh partial not exactly 0" % (R, c)
            check_chunks("gru %s R=%d TT=%d rpc=%d" % (name, R, TT, rpc), W, B, refs[i])


# ---------------------------------------------------------------------------------------------------------------------
# k_reduce_fc1
# ---------------------------------------------------------------------------------------------------------------------
def run_fc1(bs, flags, M, rpc, d_in, g):
    xs, d_x, xp = buffer2d(M, 64, 64, 0, g)
    nc = n_chunks(M, rpc)
    wb, bb = partial_buffer(nc * 64 * d_in), partial_buffer(nc * 64)
    before = nat.lib().mal_stat(b"reduce_fc1")
    nat.check(nat.lib().mal_debug_reduce_fc1(C.byref(bs), flags, xp, M, rpc, wb.data_ptr(), bb.data_ptr(),
                                             nat.current_stream()), "mal_debug_reduce_fc1")
    th.cuda.synchronize()
    assert nat.lib().mal_stat(b"reduce_fc1") == before + 1
    return take_partial(wb, (nc, 64, d_in), "fc1 part_w"), take_partial(bb, (nc, 64), "fc1 part_b"), d_x, xs


FC1_CASES = AGENT_CASES + [(20, 26, 168, 1, 0), (16, 16, 96, 1, nat.IN_NO_LAST_ACTION), (17, 4, 107, 2, nat.IN_NO_AGENT_ID)]


@pytest.mark.parametrize("vec", [True, False], ids=["vec", "scalar"])
@pytest.mark.parametrize("N,A,OBS,Bn,flags", FC1_CASES)
def test_reduce_fc1(N, A, OBS, Bn, flags, vec):
    R = Bn * N
    TT = (1500 + R - 1) // R + 1
    for M, rpc in ((TT * R, 320), (TT * R - 5, 64), (TT * R - 1, 1088)):
        g = gen(N * 31 + OBS + M + rpc)
        bs, rows, d_in, keep = agent_batch(Bn, TT, N, A, OBS, flags, M, vec, g)
        W, B, d_x, xs = run_fc1(bs, flags, M, rpc, d_in, g)
        check_chunks("fc1 M=%d rpc=%d N=%d R=%d OBS=%d d_in=%d flags=%d %s" % (M, rpc, N, R, OBS, d_in, flags,
                                                                             "vec" if vec else "scalar"),
                     W, B, chunk_sums(dy_rows(d_x), rows, M, rpc))


# ---------------------------------------------------------------------------------------------------------------------
# k_fc2_grad
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("A", [1, 11, 26, nat.MAX_ACTIONS])
@pytest.mark.parametrize("Bn,N,TT,grid", [(3, 5, 11, 1), (7, 3, 53, 5), (64, 10, 101, 601), (2, 17, 30, 3)])
def test_fc2_grad(A, Bn, N, TT, grid):
    g = gen(A * 1000 + Bn + TT + grid)
    T, R = TT - 1, Bn * N
    rows = T * R
    assert rows % (64 * grid) != 0
    actions = th.randint(0, A, (Bn, TT, N, 1), generator=g, device=DEV)
    dstore = th.full((rows + 64,), NAN, device=DEV)
    d_chosen = dstore[:rows].view(Bn, T, N)
    # live on every row, the last one included.  Positive: with A = 1 a CTA's bias partial is ONE sum of ~100 values, and
    # N(0, 1) values can cancel it to ~1e-3 of their absolute sum, where a correct fp32 sum misses the norm-wise 1e-5
    # (seen: 1.6e-5 on one CTA of 601, element-wise bar met).  h ~ N(0, 1) keeps the weight partials signed.
    d_chosen.copy_(0.5 + th.rand(Bn, T, N, generator=g, device=DEV))
    hs, h, hp = buffer2d(TT * R, 64, 64, 0, g, valid=rows)                # rows of t = T stay NaN: never read
    bs = nat.Batch(Bn, TT, N, A, 1, 1)
    bs.actions = nat.Field(actions.data_ptr(), TT * N, N)
    wb, bb = partial_buffer(grid * A * 64), partial_buffer(grid * A)
    nat.check(nat.lib().mal_debug_fc2_grad(C.byref(bs), d_chosen.data_ptr(), hp, grid, wb.data_ptr(), bb.data_ptr(),
                                           nat.current_stream()), "mal_debug_fc2_grad")
    th.cuda.synchronize()
    W = take_partial(wb, (grid, A, 64), "fc2 part_w")
    B = take_partial(bb, (grid, A), "fc2 part_b")
    check_chunks("fc2 A=%d B=%d N=%d TT=%d grid=%d" % (A, Bn, N, TT, grid), W, B, fc2_sums(d_chosen, actions, h, A, grid))


# ---------------------------------------------------------------------------------------------------------------------
# past 2^24 rows: the loaders' integer-division branch (fast_divmod is exact below 2^24 only)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M", [(1 << 24) - 1, 200 * 83887])
@pytest.mark.parametrize("flavour", [nat.RED_FFMA, nat.RED_TC3], ids=["ffma", "tc3"])
def test_state_past_2p24(flavour, M):
    T, Bn, S = 200, 83887, 8
    rpc = 16384 if flavour == nat.RED_FFMA else 113408
    try:
        g = gen(M)
        bs, state, keep = state_batch(Bn, T, S, M, S, 0, True, g)
        ys, y, yp = buffer2d(M, 16, 16, 0, g)
        (W, B), = run_generic(flavour, nat.RED_A_STATE, [dict(M=M, rpc=rpc, K=S, Nout=16, dY=y, dY_ptr=yp)], bs)
        check_chunks("state 2^24 %s M=%d rpc=%d" % (FNAME[flavour], M, rpc), W, B,
                     chunk_sums(dy_rows(y), state_rows(state, T, S), M, rpc))
    finally:
        keep = ys = y = state = bs = W = B = None
        th.cuda.empty_cache()


@pytest.mark.parametrize("kernel", ["ffma", "tc3", "fc1"])
def test_agent_input_past_2p24(kernel):
    N, OBS, A, TT, Bn = 2, 4, 3, 201, 41744
    M = TT * Bn * N
    assert M > 1 << 24
    try:
        g = gen(17)
        bs, rows, d_in, keep = agent_batch(Bn, TT, N, A, OBS, 0, M, True, g)
        if kernel == "fc1":
            rpc = 113408
            W, B, y, ys = run_fc1(bs, 0, M, rpc, d_in, g)
        else:
            flavour = nat.RED_FFMA if kernel == "ffma" else nat.RED_TC3
            rpc = 16384 if kernel == "ffma" else 113408
            ys, y, yp = buffer2d(M, 16, 16, 0, g)
            (W, B), = run_generic(flavour, nat.RED_A_AGENT_IN, [dict(M=M, rpc=rpc, K=d_in, Nout=16, dY=y, dY_ptr=yp)], bs)
        check_chunks("agent 2^24 %s M=%d rpc=%d" % (kernel, M, rpc), W, B, chunk_sums(dy_rows(y), rows, M, rpc))
    finally:
        keep = ys = y = rows = bs = W = B = None
        th.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------------------------
# rejections: non-zero, a message, and no launch
# ---------------------------------------------------------------------------------------------------------------------
def test_rejections():
    L = nat.lib()
    g = gen(0)
    p = dense_prob(100, 64, 64, 64, 0, True, g)
    keys = [b"reduce_ffma", b"reduce_tc", b"reduce_tc_swap", b"reduce_fc1"]
    wb = partial_buffer(2 * 64 * 64)
    bs, rows, d_in, keep = agent_batch(3, 4, 5, 11, 250, 0, 60, True, g)     # d_in = 266 > 256
    bs_ok, rows_ok, d_in_ok, keep_ok = agent_batch(3, 4, 5, 11, 48, 0, 60, True, g)
    x = th.zeros(64, 256, device=DEV)

    def prob(**over):
        q = dict(M=100, rows_per_chunk=64, K=64, Nout=64, shift=0, dY=p["dY_ptr"], ldy=p["dY"].stride(0), A=p["A_ptr"],
                 lda=p["lda"], part_w=wb.data_ptr(), part_b=None)
        q.update(over)
        arr = (nat.RedProb * 1)()
        arr[0] = nat.RedProb(*[q[k] for k in ("M", "rows_per_chunk", "K", "Nout", "shift", "dY", "ldy", "A", "lda",
                                              "part_w", "part_b")])
        return arr

    s = nat.current_stream()
    calls = {
        "rows_per_chunk 100": lambda: L.mal_debug_reduce(4, 0, 1, prob(rows_per_chunk=100), None, 0, s),
        "rows_per_chunk 0": lambda: L.mal_debug_reduce(0, 0, 1, prob(rows_per_chunk=0), None, 0, s),
        "rows_per_chunk -64": lambda: L.mal_debug_reduce(1, 0, 1, prob(rows_per_chunk=-64), None, 0, s),
        "null dY": lambda: L.mal_debug_reduce(4, 0, 1, prob(dY=None), None, 0, s),
        "null A": lambda: L.mal_debug_reduce(0, 0, 1, prob(A=None), None, 0, s),
        "null part_w": lambda: L.mal_debug_reduce(2, 0, 1, prob(part_w=None), None, 0, s),
        "null probs": lambda: L.mal_debug_reduce(4, 0, 1, None, None, 0, s),
        "null batch": lambda: L.mal_debug_reduce(4, 2, 1, prob(), None, 0, s),
        "flavour 5": lambda: L.mal_debug_reduce(5, 0, 1, prob(), None, 0, s),
        "fc1 d_in 266": lambda: L.mal_debug_reduce_fc1(C.byref(bs), 0, x.data_ptr(), 60, 64, wb.data_ptr(), wb.data_ptr(), s),
        "fc1 rows_per_chunk 96": lambda: L.mal_debug_reduce_fc1(C.byref(bs_ok), 0, x.data_ptr(), 60, 96, wb.data_ptr(),
                                                                wb.data_ptr(), s),
        "fc1 null d_x": lambda: L.mal_debug_reduce_fc1(C.byref(bs_ok), 0, None, 60, 64, wb.data_ptr(), wb.data_ptr(), s),
        "gru rows_per_chunk 32": lambda: L.mal_debug_reduce_gru(x.data_ptr(), x.data_ptr(), x.data_ptr(), 64, 4, 32,
                                                                *[wb.data_ptr()] * 6, s),
        "gru null x": lambda: L.mal_debug_reduce_gru(None, x.data_ptr(), x.data_ptr(), 64, 4, 64, *[wb.data_ptr()] * 6, s),
        "fc2 null d_chosen": lambda: L.mal_debug_fc2_grad(C.byref(bs_ok), None, x.data_ptr(), 4, wb.data_ptr(),
                                                          wb.data_ptr(), s),
        "fc2 grid 0": lambda: L.mal_debug_fc2_grad(C.byref(bs_ok), x.data_ptr(), x.data_ptr(), 0, wb.data_ptr(),
                                                   wb.data_ptr(), s),
    }
    th.cuda.synchronize()
    for what, call in calls.items():
        stats = [L.mal_stat(k) for k in keys]
        launches = L.mal_launch_count()
        rc = call()
        assert rc != 0, what
        msg = L.mal_last_error().decode()
        assert msg.startswith("mal_debug_"), (what, msg)
        assert L.mal_launch_count() == launches and [L.mal_stat(k) for k in keys] == stats, what
    th.cuda.synchronize()
    assert bool(th.isnan(wb).all())
