"""The kernels at the shapes where their code paths switch: large vocabularies, label sequences longer than a CTA has
threads, a non-zero blank, den graphs whose label range per CTA outgrows the shared-memory gradient accumulator.

Every case compares a CUDA entry point with a plain fp64 reference of the same operation:
  * numerator (ctc_alpha_beta_kernel / ctc_gamma_kernel) -- oracle.ctc for log p and the occupancies, and
    torch.nn.functional.ctc_loss in float64 on the CPU for log p (its gradient folds in a softmax: not the same quantity);
  * alignment (ctc_viterbi_kernel) -- a numpy Viterbi, frames in a loop, lattice cells vectorised;
  * denominator (den_backward_kernel) -- oracle.den / oracle.ctc_crf.
Tolerances as in the rest of the suite: loss 1e-4 relative, occupancies and gradients 1e-3 absolute.  bf16 inputs are
compared with the reference fed the bf16-rounded values.

Thread counts of the numerator kernels (LaunchCtcAlphaBeta / LaunchCtcViterbi): round_up(maxL + 1, 32) clamped to
[64, 1024]; thread i owns lattice cells 2i and 2i+1 and loops when maxL + 1 > 1024.  The alpha / beta passes keep the
next frame's emission row in 4 registers per thread when V <= 4 * threads and load it from global memory every frame
otherwise.  The occupancy kernel (LaunchCtcGamma) runs 8 warps per CTA while 8 * V * 4 bytes fit 48 KB and halves the
count down to 1 warp; past V = 12288 the one warp's accumulator needs more than 48 KB of dynamic shared memory.
"""
import functools

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu            # (one test here is a CPU check of the den plan: the mark is per test)

LOSS_RTOL = 1e-4
GRAD_ATOL = 1e-3
SHARED_ACC_BYTES = 64 * 1024     # den_kernels.cu LaunchDenBackward: label accumulator in shared memory up to this size


# ---------------------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=2)
def _logprobs(N, T, V, seed):
    """(N,T,V) float32 log-softmax of 3 * N(0,1) scores (cached: several cases share the large ones; treat as read-only)."""
    x = torch.randn(N, T, V, generator=torch.Generator().manual_seed(seed)) * 3.0
    return torch.log_softmax(x, -1).numpy()


def _draw_labels(rng, L, V, blank):
    """L labels from [0, V) without the blank."""
    lab = rng.integers(0, V - 1, size=L)
    lab[lab >= blank] += 1
    return lab.astype(np.int32)


def _repeats(lab):
    return int((lab[1:] == lab[:-1]).sum()) if len(lab) > 1 else 0


def _mixed_batch(V, maxL, blank=0, seed=0, extra_T=0, run_at=None, exact=False, no_skip_at=None):
    """Utterances: one at maxL labels over ~1.6 maxL frames, one short, one with L = 0; optionally (exact) the first one's
    labels again over exactly L + repeats frames (one path) and over one frame fewer (infeasible).
    run_at: a run of equal labels over positions [run_at, run_at + 10].  no_skip_at: labels[i-1] != labels[i] there."""
    rng = np.random.default_rng(seed)
    lab0 = _draw_labels(rng, maxL, V, blank)
    if run_at is not None:
        lab0[run_at:run_at + 11] = lab0[run_at]
    if no_skip_at is not None and lab0[no_skip_at] == lab0[no_skip_at - 1]:
        lab0[no_skip_at] = (lab0[no_skip_at] + 1) % V
        if lab0[no_skip_at] == blank:
            lab0[no_skip_at] = (lab0[no_skip_at] + 1) % V
        assert lab0[no_skip_at] != lab0[no_skip_at - 1]
    Ls = [maxL, min(5, maxL), 0]
    labs = [lab0, _draw_labels(rng, Ls[1], V, blank), lab0[:0]]
    lxs = [int(1.6 * maxL) + 8, 3 * Ls[1] + 4, 9]
    if exact:
        need = maxL + _repeats(lab0)
        Ls += [maxL, maxL]
        labs += [lab0, lab0]
        lxs += [need, need - 1]
    T = max(lxs) + extra_T
    y = _logprobs(len(Ls), T, V, seed)
    return (y, np.concatenate(labs).astype(np.int32), np.asarray(Ls, np.int32), np.asarray(lxs, np.int32))


def _threads(maxL):
    return min(1024, max(64, (maxL + 1 + 31) // 32 * 32))


def _row_in_regs(V, maxL):
    return V <= 4 * _threads(maxL)


def _gamma_warps(V):
    w = 8
    while w > 1 and w * V * 4 > 48 * 1024:
        w //= 2
    return w


# ---------------------------------------------------------------------------------------------------------------------
# numerator checks
# ---------------------------------------------------------------------------------------------------------------------
def _close_logp(got, ref):
    got = np.asarray(got, np.float64)
    for n in range(len(ref)):
        if np.isfinite(ref[n]):
            assert abs(got[n] - ref[n]) <= LOSS_RTOL * max(1.0, abs(ref[n])), (n, got[n], ref[n])
        else:
            assert np.isneginf(got[n]), (n, got[n])


def _num_reference(y, labels, ly, lx, blank):
    """oracle.ctc (log p, occupancies), with its log p checked against torch's fp64 CTC on the CPU."""
    from oracle import oracle
    lp, gam = oracle.ctc(y, labels, ly, lx, blank=blank)
    nll = torch.nn.functional.ctc_loss(torch.from_numpy(y).double().transpose(0, 1), torch.from_numpy(labels).long(),
                                       torch.from_numpy(lx).long(), torch.from_numpy(ly).long(), blank=blank,
                                       reduction="none", zero_infinity=False).numpy()
    _close_logp(-nll, lp)
    return lp, gam


def _check_numerator(y, labels, ly, lx, blank, dtype=torch.float32, entries=("gpu_ctc", "ctc_loss_fwd")):
    """Runs the numerator through _C.gpu_ctc ((T,N,V), host costs; with and without gradients) and _C.ctc_loss_fwd
    ((N,T,V) in place, every gradient row written) and compares both with the references."""
    from cat_b200 import _C
    N = y.shape[0]
    yk = torch.tensor(y).to(dtype)
    yr = yk.float().numpy()                                   # what the kernel sees
    lp, gam = _num_reference(yr, labels, ly, lx, blank)
    lab_t, ly_t, lx_t = torch.tensor(labels), torch.tensor(ly), torch.tensor(lx)
    if "gpu_ctc" in entries:
        act = yk.float().cuda().transpose(0, 1).contiguous()
        grads = torch.zeros_like(act)
        costs = torch.zeros(N)
        _C.gpu_ctc(act, grads, lab_t, ly_t, lx_t, N, costs, blank)
        _close_logp(costs.numpy(), lp)
        assert np.abs(grads.transpose(0, 1).cpu().numpy() - gam).max() < GRAD_ATOL
        del grads
        # costs only (no gradient buffer: the beta CTAs return at once): the same alpha pass, the same costs
        costs_only = torch.zeros(N)
        _C.gpu_ctc(act, torch.empty(0, device="cuda"), lab_t, ly_t, lx_t, N, costs_only, blank)
        assert torch.equal(costs_only, costs), (costs_only, costs)
        del act
    if "ctc_loss_fwd" in entries:
        loss, grad, logp = _C.ctc_loss_fwd(yk.cuda(), lab_t, lx_t, ly_t, size_average=False, blank=blank)
        _close_logp(logp.cpu().numpy(), lp)
        assert np.abs(-grad.cpu().numpy() - gam).max() < GRAD_ATOL
        total = -lp.sum()
        if np.isfinite(total):
            assert abs(float(loss) - total) <= LOSS_RTOL * max(1.0, abs(total))
        else:
            assert float(loss) == np.inf
    return lp


# ---- vocabulary against the register row ------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("V,maxL", [
    pytest.param(256, 30, id="maxL30-64thr-V256-last-row-in-regs(4x64=256)"),
    pytest.param(257, 30, id="maxL30-64thr-V257-first-global-row(257>4x64)"),
    pytest.param(1000, 30, id="maxL30-64thr-V1000-global-row"),
    pytest.param(5000, 63, id="maxL63-64thr-V5000-global-row"),
    pytest.param(4096, 1023, id="maxL1023-1024thr-V4096-last-row-in-regs(4x1024)"),
    pytest.param(4097, 1023, id="maxL1023-1024thr-V4097-first-global-row"),
])
def test_numerator_vocab_vs_register_row(V, maxL):
    """maxL <= 63: round_up(maxL+1, 32) <= 64 -> 64 threads -> rows in registers only for V <= 256.
    maxL = 1023: 1024 threads -> rows in registers only for V <= 4096."""
    assert _row_in_regs(V, maxL) == (V in (256, 4096))
    y, labels, ly, lx = _mixed_batch(V, maxL, seed=V + maxL)
    _check_numerator(y, labels, ly, lx, 0)


# ---- label length against the thread count -----------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("maxL", [
    pytest.param(63, id="maxL63-L1=64-64thr-one-pair-each"),
    pytest.param(64, id="maxL64-L1=65-96thr"),
    pytest.param(1023, id="maxL1023-L1=1024-1024thr-one-pair-each"),
    pytest.param(1024, id="maxL1024-L1=1025>1024thr-thread0-wraps-to-final-blank-cell-2048"),
    pytest.param(1100, id="maxL1100-threads-capped-1024-label-skip-from-pair1023-into-pair1024"),
    pytest.param(1500, id="maxL1500-threads-capped-1024-repeat-run-1020..1030-across-wrap-exact-and-short-utts"),
])
def test_numerator_label_length_vs_threads(maxL):
    """Cells 2i, 2i+1 belong to thread i mod 1024: past 1023 label positions the cell loops wrap around, and the skip rule
    (no skip into a label equal to the previous one) reads s_lab[i-1] written by another thread's iteration.  V = 40, rows
    in registers.  maxL = 1500 also carries the first utterance's labels over exactly L + repeats frames (one path:
    occupancies 0/1) and over one frame fewer (infeasible: log p = -inf, no gradient)."""
    kw = {}
    if maxL == 1100:
        kw["no_skip_at"] = 1024                     # a skip transition from pair 1023 (thread 1023) into pair 1024 (thread 0)
    if maxL == 1500:
        kw.update(run_at=1020, exact=True)
    y, labels, ly, lx = _mixed_batch(40, maxL, seed=maxL, **kw)
    if maxL == 1500:
        assert (labels[1020:1031] == labels[1020]).all() and lx[3] == maxL + _repeats(labels[:maxL]) and lx[4] == lx[3] - 1
    lp = _check_numerator(y, labels, ly, lx, 0)
    if maxL == 1500:
        assert np.isfinite(lp[3]) and np.isneginf(lp[4])


# ---- occupancy kernel CTA shapes -----------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("V", [
    pytest.param(1536, id="V1536-8warps(8x1536x4=48KB)"),
    pytest.param(1537, id="V1537-4warps(<8-warps-per-CTA)"),
    pytest.param(6144, id="V6144-2warps(2x6144x4=48KB)"),
    pytest.param(6145, id="V6145-1warp"),
    pytest.param(12289, id="V12289-1warp-over-48KB-dynamic-smem(12289x4)"),
    pytest.param(16000, id="V16000-1warp-64000B-dynamic-smem"),
])
def test_numerator_occupancy_cta_shapes(V):
    """LaunchCtcGamma: warps per CTA = 8 halved while warps * V * 4 > 48 KB (down to 1, with > 48 KB opted in)."""
    assert _gamma_warps(V) == {1536: 8, 1537: 4, 6144: 2, 6145: 1, 12289: 1, 16000: 1}[V]
    y, labels, ly, lx = _mixed_batch(V, 10, seed=V)
    _check_numerator(y, labels, ly, lx, 0)


# ---- shared-memory limit of the numerator -------------------------------------------------------------------------------
def _numerator_smem(maxL, V):
    """LaunchCtcAlphaBeta's request: a[2][2maxL+1] doubles | lab[maxL+1] ints | yrow[2][V] floats | 16."""
    return 2 * (2 * maxL + 1) * 8 + (maxL + 1) * 4 + 2 * V * 4 + 16


@gpu
def test_numerator_shared_memory_limit():
    """The numerator stages two emission rows in shared memory and refuses requests over 200 KB on the host, before any
    launch: with maxL = 10 that is 396 + 8 V bytes, so V = 25550 is the largest vocabulary it runs.  Below the limit it
    matches the oracle; past it both entry points raise, and the process goes on computing correct results."""
    from cat_b200 import _C
    limit = 200 * 1024
    assert _numerator_smem(10, 25550) <= limit < _numerator_smem(10, 25551)
    for V in (25000, 25550):
        y, labels, ly, lx = _mixed_batch(V, 10, seed=V)
        _check_numerator(y, labels, ly, lx, 0)
    msg = "too long for the numerator kernel's shared memory"
    for V in (25551, 26000):
        y, labels, ly, lx = _mixed_batch(V, 10, seed=V)
        lab_t, ly_t, lx_t = torch.tensor(labels), torch.tensor(ly), torch.tensor(lx)
        with pytest.raises(RuntimeError, match=msg):
            _C.ctc_loss_fwd(torch.tensor(y, device="cuda"), lab_t, lx_t, ly_t, size_average=True)
        act = torch.tensor(y, device="cuda").transpose(0, 1).contiguous()
        with pytest.raises(RuntimeError, match=msg):
            _C.gpu_ctc(act, torch.zeros_like(act), lab_t, ly_t, lx_t, len(ly), torch.zeros(len(ly)), 0)
        del act
    y, labels, ly, lx = _mixed_batch(1000, 30, seed=7)
    _check_numerator(y, labels, ly, lx, 0)


# ---- non-zero blank -------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("V,blank", [
    pytest.param(40, 1, id="V40-maxL30-rows-in-regs-blank1"),
    pytest.param(40, 39, id="V40-maxL30-rows-in-regs-blank=V-1"),
    pytest.param(1000, 1, id="V1000-maxL30-global-row(1000>4x64)-blank1"),
    pytest.param(1000, 999, id="V1000-maxL30-global-row-blank=V-1"),
])
def test_numerator_nonzero_blank(V, blank):
    """blank_label of gpu_ctc / blank of ctc_loss_fwd: the blank cells of all three numerator kernels read column
    `blank`, and labels are drawn from [0, V) without it (label 0 is an ordinary token here)."""
    y, labels, ly, lx = _mixed_batch(V, 30, blank=blank, seed=blank)
    assert not (labels == blank).any()
    _check_numerator(y, labels, ly, lx, blank)


# ---- bf16 logits through the CTC-only loss -----------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("V,maxL", [
    pytest.param(200, 30, id="bf16-V200-maxL30-rows-in-regs"),
    pytest.param(1000, 30, id="bf16-V1000-maxL30-global-row"),
    pytest.param(300, 1500, id="bf16-V300-maxL1500-1024thr-wrap"),
])
def test_ctc_loss_fwd_bf16(V, maxL):
    y, labels, ly, lx = _mixed_batch(V, maxL, seed=3 * V + maxL)
    _check_numerator(y, labels, ly, lx, 0, dtype=torch.bfloat16, entries=("ctc_loss_fwd",))


# ---- padded frames in the CTC-only loss ---------------------------------------------------------------------------------
@gpu
def test_ctc_loss_fwd_writes_padding_rows():
    """T = max(lx) + 17: the gradient comes from torch.empty and the occupancy kernel (overwrite mode) must write rows
    [max(lx), T) -- and every row t >= lx[n] -- as zeros.  The gradient is placed on a block filled with NaN first.
    (V = 2000: the gradient's 1.75 MB come from the caching allocator's large-block pool, which the small label upload
    before it does not touch, so the freed NaN block is the one handed out next.)"""
    from cat_b200 import _C
    V = 2000
    y, labels, ly, lx = _mixed_batch(V, 30, seed=17, extra_T=17)
    N, T, _ = y.shape
    assert T == lx.max() + 17
    lp, gam = _num_reference(y, labels, ly, lx, 0)
    logits = torch.tensor(y, device="cuda")
    lab_t, ly_t, lx_t = torch.tensor(labels), torch.tensor(ly), torch.tensor(lx)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    poison = torch.full((N * T * V,), float("nan"), dtype=torch.float32, device="cuda")
    ptr = poison.data_ptr()
    del poison
    loss, grad, logp = _C.ctc_loss_fwd(logits, lab_t, lx_t, ly_t, size_average=False)
    assert grad.data_ptr() == ptr, "the gradient did not reuse the NaN-filled block: this test would prove nothing"
    g = grad.cpu().numpy()
    for n in range(N):
        assert (g[n, lx[n]:] == 0).all(), n
    assert not np.isnan(g).any()
    _close_logp(logp.cpu().numpy(), lp)
    assert np.abs(-g - gam).max() < GRAD_ATOL


# ---- fused loss with a long label sequence ------------------------------------------------------------------------------
@gpu
def test_fused_loss_long_labels(tmp_graphs):
    """CTC_CRF_LOSS with maxL = 1100 (threads capped at 1024, cell loops wrap) over ~1800 frames: the fused call keeps the
    numerator's log-likelihoods behind a [N][2][T][2 maxL + 1]-double cell workspace (LossFwdImpl `logp`)."""
    import ctc_crf
    from oracle import oracle
    path, g, V = tmp_graphs["tlm_mid"]
    rng = np.random.default_rng(11)
    ly = np.array([1100, 300, 0], np.int32)
    lx = np.array([1800, 700, 40], np.int32)
    labels = np.concatenate([rng.integers(1, V, size=int(L)) for L in ly]).astype(np.int32)
    y = _logprobs(3, 1800, V, 11)
    ctx = ctc_crf.CRFContext(path, gpus=0)
    logits = torch.tensor(y, device="cuda").requires_grad_(True)
    loss = ctc_crf.CTC_CRF_LOSS(lamb=0.1)(logits, torch.tensor(labels), torch.tensor(lx), torch.tensor(ly))
    loss.backward()
    oloss, ograd, _ = oracle.ctc_crf(g, y, labels, lx, ly, 0.1)
    assert np.isfinite(oloss)
    assert abs(loss.item() - oloss) <= LOSS_RTOL * max(1.0, abs(oloss)), (loss.item(), oloss)
    assert np.abs(logits.grad.cpu().numpy() - ograd).max() < GRAD_ATOL
    del ctx


# ---------------------------------------------------------------------------------------------------------------------
# alignment
# ---------------------------------------------------------------------------------------------------------------------
def _viterbi_np(y, lab, blank):
    """Best path over the blank-expanded lattice in fp64, one frame at a time, cells vectorised.  Ties go to the smaller
    predecessor offset (stay < s-1 < s-2).  Returns (token per frame, score); score -inf if there is no path."""
    T = y.shape[0]
    ext = np.full(2 * len(lab) + 1, blank, np.int64)
    ext[1::2] = lab
    S = ext.size
    skip = np.zeros(S, bool)
    skip[2:] = (ext[2:] != blank) & (ext[2:] != ext[:-2])
    emit = y[:, ext]
    v = np.full(S, -np.inf)
    v[0] = emit[0, 0]
    if S > 1:
        v[1] = emit[0, 1]
    bp = np.zeros((T, S), np.int8)
    c1 = np.empty(S)
    c2 = np.empty(S)
    for t in range(1, T):
        best = v.copy()
        k = np.zeros(S, np.int8)
        c1[0] = -np.inf
        c1[1:] = v[:-1]
        m = c1 > best
        best[m] = c1[m]
        k[m] = 1
        c2[:2] = -np.inf
        c2[2:] = np.where(skip[2:], v[:-2], -np.inf)
        m = c2 > best
        best[m] = c2[m]
        k[m] = 2
        v = best + emit[t]
        bp[t] = k
    s = S - 1
    if S > 1 and v[S - 2] > v[S - 1]:
        s = S - 2
    score = v[s]
    path = np.empty(T, np.int64)
    if not np.isfinite(score):
        return path, score
    for t in range(T - 1, -1, -1):
        path[t] = ext[s]
        s -= int(bp[t, s])
    assert s in (0, 1)
    return path, score


def _collapse(path, blank):
    return [int(k) for i, k in enumerate(path) if k != blank and (i == 0 or path[i - 1] != k)]


@gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("blank", [0, 4999], ids=["blank0", "blank=V-1"])
def test_ctc_align_long_labels_large_vocab(blank, dtype):
    """_C.ctc_align at maxL = 1500 (threads capped at 1024: cell loops wrap, a repeat run over positions 1020..1030) and
    V = 5000 with the blank at 0 or V-1; plus a short, an empty, an exactly feasible (L + repeats frames) and an
    infeasible (one frame fewer) utterance."""
    from cat_b200 import _C
    V, maxL = 5000, 1500
    y, labels, ly, lx = _mixed_batch(V, maxL, blank=blank, seed=5, run_at=1020, exact=True)
    yk = torch.tensor(y).to(dtype)
    yr = yk.float().numpy().astype(np.float64)
    align, score = _C.ctc_align(yk.cuda(), torch.tensor(labels), torch.tensor(lx), torch.tensor(ly), blank=blank)
    align, score = align.cpu().numpy(), score.cpu().numpy()
    off = np.concatenate([[0], np.cumsum(ly)])
    for n in range(len(ly)):
        lab = labels[off[n]:off[n + 1]]
        ref, sc = _viterbi_np(yr[n, :lx[n]], lab, blank)
        assert (align[n, lx[n]:] == -1).all(), n
        if not np.isfinite(sc):
            assert n == 4 and np.isneginf(score[n]) and (align[n] == -1).all()
            continue
        got = align[n, :lx[n]]
        assert abs(score[n] - sc) <= LOSS_RTOL * max(1.0, abs(sc)), (n, score[n], sc)
        # the returned path's own score, recomputed in fp64; a different path is accepted only as a tie
        own = float(yr[n, np.arange(lx[n]), got].sum())
        if not np.array_equal(got, ref):
            assert abs(own - sc) <= LOSS_RTOL * max(1.0, abs(sc)), (n, own, sc)
        assert _collapse(got, blank) == [int(k) for k in lab], n
        if n == 3:                               # L + repeats frames: the only path, one frame per label and separating blank
            assert np.array_equal(got, ref)


# ---------------------------------------------------------------------------------------------------------------------
# denominator at a large vocabulary
# ---------------------------------------------------------------------------------------------------------------------
def _pad_lanes(N):
    """common.cuh PadLanes for N > 16: whole 32-lane groups, 1, 2 or a multiple of 4 of them."""
    assert N > 16
    g = (N + 31) // 32
    if g >= 3:
        g = (g + 3) // 4 * 4
    return g * 32


def _max_tile_labels(pv):
    cl = pv.bwd.cta_labels
    return int((cl[:, 1] + cl[:, 3]).max())


@pytest.fixture(scope="module")
def big_graphs(tmp_path_factory):
    """T-compose-LM shaped den graphs with one token per LM history: H = V = 8000 and 40000 (about 5 000 / 25 000 labels
    in use, 88 k / 440 k arcs)."""
    from cat_b200 import fst
    d = tmp_path_factory.mktemp("big_graphs")
    out = {}
    for H in (8000, 40000):
        g = fst.make_synthetic_den(H, 4, H, seed=7)
        path = str(d / f"tlm_{H}.fst")
        fst.write_fst(path, g)
        out[H] = (path, g)
    return out


# den graph, batch width of the GPU test that relies on the direct-atomic branch
DIRECT_ATOMIC_CASES = [(8000, 130), (40000, 64)]


def test_den_direct_atomic_branch_is_reached(big_graphs):
    """CPU: LaunchDenBackward keeps the gradient's label accumulator in shared memory only while
    max_tile_labels * PadLanes(N) * 4 <= 64 KB.  On the B200 plan (148 CTAs x 16 warps) the 8000-label graph exceeds that
    at 256 lanes (N = 129..256) and the 40000-label graph at 64 lanes (N = 33..64), so the GPU tests below run
    den_backward_kernel's direct global atomics.  If a plan change packs the labels tighter, this fails instead of the GPU
    tests silently going back to the shared accumulator."""
    from cat_b200 import plan
    for H, N in DIRECT_ATOMIC_CASES:
        pv = plan.load_plan(big_graphs[H][0], 148, 16)
        m = _max_tile_labels(pv)
        assert m * _pad_lanes(N) * 4 > SHARED_ACC_BYTES, (H, N, m)
        if H == 8000:                 # ... while 64 lanes (the fused loss's default slice) still use the accumulator
            assert m * 64 * 4 <= SHARED_ACC_BYTES, m


def _ctx(path):
    import ctc_crf
    return ctc_crf.CRFContext(path, gpus=0)


def _device_plan_direct_atomic(path, N):
    from cat_b200 import plan
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    pv = plan.load_plan(path, sms, 16)
    assert _max_tile_labels(pv) * _pad_lanes(N) * 4 > SHARED_ACC_BYTES, "direct-atomic branch not reached on this device"
    return pv


def _den_run(y, lens):
    from cat_b200 import _C
    logits = torch.tensor(y, device="cuda")
    grad = torch.zeros_like(logits)
    N = y.shape[0]
    ca, cb = torch.zeros(N, device="cuda"), torch.zeros(N, device="cuda")
    _C.gpu_den(logits, grad, torch.tensor(lens, dtype=torch.int32).cuda(), ca, cb)
    return ca.cpu().numpy(), cb.cpu().numpy(), grad.cpu().numpy()


def _pick(lens):
    """longest, shortest and two middle utterances"""
    o = np.argsort(lens, kind="stable")
    return sorted({int(o[-1]), int(o[0]), int(o[len(o) // 2]), int(o[len(o) // 2 + 1])})


@gpu
@pytest.mark.parametrize("H,N", [
    pytest.param(8000, 130, id="H8000-N130-256lanes-79labels/tile(x256x4>64KB)-direct-atomics"),
    pytest.param(40000, 64, id="H40000-N64-64lanes-over-256labels/tile(x64x4>64KB)-direct-atomics"),
])
def test_den_large_vocab_direct_atomics(big_graphs, H, N):
    """_C.gpu_den where a CTA's label range does not fit the 64 KB shared accumulator (flush_gsum's global-atomic
    branch): logZ from alpha and beta and the occupancies against oracle.den on the longest, the shortest and two middle
    utterances; rows past each length stay zero.  The 8000 graph is run again as a 16-utterance batch (small-batch tier,
    shared accumulator): per utterance the two runs agree to 1e-5."""
    from oracle import oracle
    path, g = big_graphs[H]
    pv = _device_plan_direct_atomic(path, N)
    V = pv.num_labels
    T = 16
    lens = np.maximum(1, T - (np.arange(N) * 5) % T).astype(np.int32)
    lens[0] = T
    y = _logprobs(N, T, V, H)
    ctx = _ctx(path)
    ca, cb, gn = _den_run(y, lens)
    sel = _pick(lens)
    la, lb, gd = oracle.den(g, y[sel], lens[sel], fast=True)
    np.testing.assert_allclose(ca[sel], la, rtol=LOSS_RTOL, atol=1e-4)
    np.testing.assert_allclose(cb[sel], lb, rtol=LOSS_RTOL, atol=1e-4)
    assert np.abs(gn[sel] - gd).max() < GRAD_ATOL
    for n in range(N):
        assert not gn[n, lens[n]:].any()
    if H == 8000:
        others = [n for n in range(0, N, 7) if n not in sel]
        sub = sorted(set(sel) | set(others[:16 - len(sel)]))
        assert len(sub) == 16
        assert _max_tile_labels(pv) * 32 * 4 <= SHARED_ACC_BYTES     # 16- or 32-lane padding: shared accumulator
        ca16, cb16, g16 = _den_run(np.ascontiguousarray(y[sub]), lens[sub])
        np.testing.assert_allclose(ca16, ca[sub], rtol=1e-5, atol=1e-5)
        np.testing.assert_allclose(cb16, cb[sub], rtol=1e-5, atol=1e-5)
        assert np.abs(g16 - gn[sub]).max() < 1e-5
        pos = [sub.index(n) for n in sel]
        assert np.abs(g16[pos] - gd).max() < GRAD_ATOL
    del ctx


@gpu
def test_fused_loss_direct_atomics(big_graphs, monkeypatch):
    """CTC_CRF_LOSS itself through the direct-atomic den branch: 130 utterances in one call (slice width raised from 64 to
    256) on the 8000 graph -> 256 lanes, 79 labels per tile x 256 x 4 > 64 KB.  Per-utterance parts and gradient rows of
    four utterances against oracle.ctc_crf, the loss against the sum of the parts."""
    from cat_b200 import _C
    from oracle import oracle
    path, g = big_graphs[8000]
    N, T, lamb = 130, 16, 0.1
    pv = _device_plan_direct_atomic(path, N)
    V = pv.num_labels
    monkeypatch.setattr(_C, "MAX_UTTS_PER_CALL", 256)
    rng = np.random.default_rng(13)
    lens = np.maximum(2, T - (np.arange(N) * 3) % T).astype(np.int32)
    ly = np.maximum(0, lens // 3 - 1).astype(np.int32)
    labels = rng.integers(1, V, size=int(ly.sum())).astype(np.int32)
    y = _logprobs(N, T, V, 8000)
    ctx = _ctx(path)
    loss, grad, parts = _C.ctc_crf_loss_fwd(torch.tensor(y, device="cuda"), torch.tensor(labels), torch.tensor(lens),
                                            torch.tensor(ly), lamb, False, want_parts=True)
    parts = parts.cpu().numpy().astype(np.float64)
    total = (parts[:N] - (1 + lamb) * parts[N:]).sum()
    assert abs(float(loss) - total) <= LOSS_RTOL * max(1.0, abs(total))
    sel = _pick(lens)
    off = np.concatenate([[0], np.cumsum(ly)])
    sub_labels = np.concatenate([labels[off[n]:off[n + 1]] for n in sel]).astype(np.int32)
    oloss, ograd, op = oracle.ctc_crf(g, y[sel], sub_labels, lens[sel], ly[sel], lamb, size_average=False, fast=True)
    np.testing.assert_allclose(parts[sel], op["logz_alpha"], rtol=LOSS_RTOL, atol=1e-4)
    np.testing.assert_allclose(parts[N + np.asarray(sel)], op["logp_ctc"], rtol=LOSS_RTOL, atol=1e-4)
    assert np.abs(grad.cpu().numpy()[sel] - ograd).max() < GRAD_ATOL
    del ctx


@gpu
def test_fused_loss_past_numerator_vocab_limit(big_graphs):
    """The fused loss at 64 lanes would take the direct-atomic den branch only past ~256 labels per tile, i.e. with the
    40000 graph; its ~40 000 classes exceed what the numerator stages in shared memory (2 rows x V x 4 bytes within
    200 KB: V <= 25 550 at short labels).  The call raises that limit's error; it does not compute a wrong loss."""
    import ctc_crf
    path, g = big_graphs[40000]
    pv = _device_plan_direct_atomic(path, 64)
    V, T, N = pv.num_labels, 4, 2
    assert _numerator_smem(2, V) > 200 * 1024
    ctx = _ctx(path)
    y = torch.log_softmax(torch.randn(N, T, V, generator=torch.Generator().manual_seed(1)), -1).cuda()
    with pytest.raises(RuntimeError, match="too long for the numerator kernel's shared memory"):
        ctc_crf.CTC_CRF_LOSS()(y, torch.tensor([1, 2, 3], dtype=torch.int32), torch.tensor([T, T], dtype=torch.int32),
                               torch.tensor([2, 1], dtype=torch.int32))
    del ctx


@gpu
@pytest.mark.parametrize("from_logits", [False, True], ids=["logprobs", "from_logits"])
def test_fused_loss_columns_past_graph_labels(big_graphs, from_logits):
    """Logits with 37 columns past the den graph's labels, holding each frame's maximum + 5 nats: frame_max_kernel takes
    its shift from a column the recursion never reads.  Log-prob input: the extra columns get exactly zero gradient.
    Raw-logit input: they get the softmax term of the log_softmax Jacobian (not zero) -- against the oracle either way."""
    import ctc_crf
    from oracle import oracle
    path, g = big_graphs[8000]
    N, T, lamb = 8, 16, 0.1
    ctx = _ctx(path)
    Vg = int(g.ilabel.max())                 # the graph's labels are ilabel - 1 in [0, Vg)
    V = Vg + 37
    rng = np.random.default_rng(21)
    lens = np.array([16, 16, 14, 11, 9, 6, 3, 1], np.int32)
    ly = (lens // 3).astype(np.int32)
    labels = rng.integers(1, Vg, size=int(ly.sum())).astype(np.int32)
    y = np.empty((N, T, V), np.float32)
    y[..., :Vg] = _logprobs(N, T, Vg, 21)
    y[..., Vg:] = y[..., :Vg].max(-1, keepdims=True) + 5.0
    logits = torch.tensor(y, device="cuda").requires_grad_(True)
    loss = ctc_crf.CTC_CRF_LOSS(lamb=lamb, from_logits=from_logits)(logits, torch.tensor(labels), torch.tensor(lens),
                                                                   torch.tensor(ly))
    loss.backward()
    gr = logits.grad.cpu().numpy()
    if from_logits:
        oloss, ograd, _ = oracle.ctc_crf_from_logits(g, y, labels, lens, ly, lamb)
        # -softmax(z) * sum_k g_k: about lamb / N / 37 = 3e-4, under the gradient tolerance, so checked relative to itself
        valid = np.arange(T)[None, :] < lens[:, None]
        ex, oex = gr[..., Vg:][valid], ograd[..., Vg:][valid]
        assert (ex != 0).all() and (np.abs(ex - oex) <= 5e-2 * np.abs(oex) + 1e-6).all()
    else:
        oloss, ograd, _ = oracle.ctc_crf(g, y, labels, lens, ly, lamb, fast=True)
        assert (gr[..., Vg:] == 0).all()
    assert abs(loss.item() - oloss) <= LOSS_RTOL * max(1.0, abs(oloss)), (loss.item(), oloss)
    assert np.abs(gr - ograd).max() < GRAD_ATOL
    del ctx
