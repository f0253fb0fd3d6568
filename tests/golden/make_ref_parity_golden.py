"""Records what tests/test_gpu_parity.py compares against from the REFERENCE'S OWN CUDA CODE (oracle/_ref, the sm100fix
build of oracle/Makefile), so that those tests need neither the reference sources nor its build.  Needs a GPU and
oracle/_ref built; writes OUTDIR/ref_cuda_parity.npz (default: next to this script):

    python tests/golden/make_ref_parity_golden.py [OUTDIR]

Two cases, on the tests' own seeded inputs:
  t120  test_vs_reference_cuda:     V=218, 100k-arc graph, N=8, T=120
  t800  test_full_size_properties:  V=218, 1M-arc graph, N=32, T=800
Per case: the reference's loss, its gradient on a fixed seeded sample of (utterance, frame) rows (the whole gradient is
several MB), and fingerprints of the inputs.  t800 also keeps the reference's distance from the fp64 oracle on
utterances 0 and N-1 and the largest error of its gradient row sums.
"""
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from cat_b200 import fst  # noqa: E402
from oracle import oracle, ref_cuda  # noqa: E402


def sample_rows(lens, per_utt, seed):
    """Sorted (utterance, frame) pairs: `per_utt` distinct valid frames of every utterance."""
    rng = np.random.default_rng(seed)
    return np.array([(n, t) for n, L in enumerate(lens) for t in np.sort(rng.choice(int(L), per_utt, replace=False))],
                    np.int32)


def fingerprint(g, y, labels):
    return dict(num_arcs=np.array(g.num_arcs), y_sum=np.array(np.float64(y).sum()),
                labels_sum=np.array(int(np.int64(labels).sum())))


def reference(path, y, labels, lens, ly, lamb):
    ctx = ref_cuda.RefContext(path, 0)
    loss, grad, parts = ref_cuda.ctc_crf_forward(ctx, torch.tensor(y, device="cuda"), torch.tensor(labels),
                                                 torch.tensor(lens), torch.tensor(ly), lamb, True)
    torch.cuda.synchronize()
    ctx.close()
    assert parts["ctc_status"] == 0, parts["ctc_status"]
    return float(loss.item()), grad.cpu().numpy()


def main(outdir):
    assert ref_cuda.available(), "oracle/_ref is not built"
    out = {}
    V, lamb = 218, 0.01
    tmpdir = tempfile.TemporaryDirectory(prefix="ccb_golden_")
    tmp = os.path.join(tmpdir.name, "den.fst")

    g = fst.make_synthetic_den(2000, 24, V, seed=7)
    fst.write_fst(tmp, g)
    y, labels, lens, ly = oracle.synth_batch(8, 120, V, seed=1234, lens=[120, 120, 111, 97, 80, 64, 30, 12])
    loss, grad = reference(tmp, y, labels, lens, ly, lamb)
    rows = sample_rows(lens, 8, seed=120)
    out.update({f"t120/{k}": v for k, v in fingerprint(g, y, labels).items()})
    out.update({"t120/loss": np.array(loss), "t120/rows": rows, "t120/grad_rows": grad[rows[:, 0], rows[:, 1]]})
    print("t120 reference loss", loss)

    g = fst.make_synthetic_den(20000, 24, V, seed=7)
    fst.write_fst(tmp, g)
    N = 32
    y, labels, lens, ly = oracle.synth_batch(N, 800, V, seed=1234)
    loss, grad = reference(tmp, y, labels, lens, ly, lamb)
    rows = sample_rows(lens, 1, seed=800)
    sub = [0, N - 1]
    off = np.concatenate([[0], np.cumsum(ly)])
    sub_labels = np.concatenate([labels[off[i]:off[i + 1]] for i in sub])
    _, ograd, _ = oracle.ctc_crf(g, y[sub], sub_labels, lens[sub], ly[sub], lamb, size_average=False, nthreads=2)
    out.update({f"t800/{k}": v for k, v in fingerprint(g, y, labels).items()})
    out.update({"t800/loss": np.array(loss), "t800/rows": rows, "t800/grad_rows": grad[rows[:, 0], rows[:, 1]],
                "t800/ref_vs_oracle": np.array(np.abs(grad[sub] * N - ograd).max()),
                "t800/ref_row_sum_err": np.array(np.abs(grad.sum(-1) * N + lamb).max())})
    print("t800 reference loss", loss, "| max |reference - oracle|:", float(out["t800/ref_vs_oracle"]))
    tmpdir.cleanup()

    path = os.path.join(outdir, "ref_cuda_parity.npz")
    np.savez_compressed(path, **out)
    print("wrote", path)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.dirname(os.path.abspath(__file__)))
