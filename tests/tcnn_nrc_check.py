#!/usr/bin/env python
"""Pins the NRC network (SURVEY.md §8a rows N4-N6) against the reference's own code: tiny-cuda-nn's NetworkWithInputEncoding +
Trainer built from neural_radiance_caching/network_interface.cu's config, compiled from the reference's vendored tiny-cuda-nn
into oracle/_ref/libtcnn_nrc.so (oracle/ref_tcnn/tcnn_nrc.cu, Makefile).  Runs on a GPU in its own process (the live check
launches third-party kernels: a fault there must not take the test session's CUDA context with it) and prints ONE JSON line:

  init        tcnn's pcg32{1337} initial parameters vs gfx_nrc_create's (bit-exact fp32 master weights wanted)
  forward     relative L2 of the inferred radiance: this repo's tcgen05 kernel / the oracle (fp32 and half accumulation) vs tcnn
  gradients   one training step from identical weights: relative L2 per weight matrix and for the hash grid, same three arms
  weights     training / inference (EMA) weights after four training steps
  timing      ms per call of tcnn's own launches and of this repo's, same B200, same inputs (2 116 608 queries; 16 384 samples)

  python tests/tcnn_nrc_check.py [--no-timing]           live: runs tiny-cuda-nn (oracle/_ref/libtcnn_nrc.so)
  python tests/tcnn_nrc_check.py --write-golden PATH     live, and stores tiny-cuda-nn's outputs in PATH (.npz)
  python tests/tcnn_nrc_check.py --golden PATH           against the stored outputs: no oracle/_ref needed, no timing

The stored outputs are a fixed, seeded sample (GOLDEN_ROWS rows of each inference, GOLDEN_PARAMS entries of each weight matrix
and of the hash grid) so that the file stays small; the initial parameters, which must match bit for bit, are kept as SHA-256
digests of all of them.  The relative L2 errors of the golden check are taken over that sample."""
import argparse
import ctypes as C
import hashlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch

import oracle_lib as O
from gfxexp_b200 import abi, engine

HIDDEN, LR = 2, 1e-2  # neural_radiance_caching_main.cpp:458-460
N_INF, N_TR = 128 * 256, 16384
GOLDEN_ROWS, GOLDEN_PARAMS = 1024, {"W0": 1024, "W1": 1024, "W2": 1024, "grid": 2048}


class TcnnNrc:
    def __init__(self):
        self.lib = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libtcnn_nrc.so"))
        vp, u32 = C.c_void_p, C.c_uint32
        L = self.lib
        L.tcnn_nrc_last_error.restype = C.c_char_p
        L.tcnn_nrc_create.argtypes = [u32, u32, C.c_float, C.POINTER(vp)]
        L.tcnn_nrc_destroy.argtypes = [vp]
        L.tcnn_nrc_num_params.argtypes = [vp]
        L.tcnn_nrc_num_params.restype = u32
        L.tcnn_nrc_read.argtypes = [vp, C.c_int, vp]
        L.tcnn_nrc_set_params.argtypes = [vp, vp]
        L.tcnn_nrc_infer.argtypes = [vp, vp, u32, vp]
        L.tcnn_nrc_train.argtypes = [vp, vp, vp, u32, C.POINTER(C.c_float)]
        L.tcnn_nrc_forward_backward.argtypes = [vp, vp, vp, u32, C.POINTER(C.c_float), vp]
        L.tcnn_nrc_time_infer.argtypes = [vp, vp, u32, u32, u32, C.POINTER(C.c_float)]
        L.tcnn_nrc_time_train.argtypes = [vp, vp, vp, u32, u32, u32, C.POINTER(C.c_float)]
        self.h = vp()
        self._ok(L.tcnn_nrc_create(1, HIDDEN, LR, C.byref(self.h)))  # 1 = PositionEncoding::HashGrid
        self.num_params = L.tcnn_nrc_num_params(self.h)

    def _ok(self, rc):
        if rc != 0:
            raise RuntimeError("tiny-cuda-nn: " + self.lib.tcnn_nrc_last_error().decode())

    def read(self, which):
        out = np.empty(self.num_params, dtype=np.float32 if which == 0 else np.float16)
        self._ok(self.lib.tcnn_nrc_read(self.h, which, out.ctypes.data))
        return out

    def set_params(self, master):
        m = np.ascontiguousarray(master, dtype=np.float32)
        self._ok(self.lib.tcnn_nrc_set_params(self.h, m.ctypes.data))

    def infer(self, q):
        out = np.empty((q.shape[0], 3), dtype=np.float32)
        self._ok(self.lib.tcnn_nrc_infer(self.h, q.ctypes.data, q.shape[0], out.ctypes.data))
        return out

    def train(self, q, t):
        loss = C.c_float()
        self._ok(self.lib.tcnn_nrc_train(self.h, q.ctypes.data, t.ctypes.data, q.shape[0], C.byref(loss)))
        return loss.value

    def forward_backward(self, q, t):
        loss = C.c_float()
        self._ok(self.lib.tcnn_nrc_forward_backward(self.h, q.ctypes.data, t.ctypes.data, q.shape[0], C.byref(loss), None))
        return loss.value, self.read(3).astype(np.float32)

    def time_infer(self, q, warmup, iters):
        ms = C.c_float()
        self._ok(self.lib.tcnn_nrc_time_infer(self.h, q.ctypes.data, q.shape[0], warmup, iters, C.byref(ms)))
        return ms.value

    def time_train(self, q, t, warmup, iters):
        ms = C.c_float()
        self._ok(self.lib.tcnn_nrc_time_train(self.h, q.ctypes.data, t.ctypes.data, q.shape[0], warmup, iters, C.byref(ms)))
        return ms.value


def rel_l2(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def queries(rng, n):
    """radiance queries as createRadianceQuery writes them (optix_pathtracing_kernels.cu:12-34): position in the unit cube,
    polar angles, 1 - exp(-roughness), reflectances - everything in [0, 1] but the angles, which span [-pi, pi] / [0, pi]"""
    q = rng.uniform(0.0, 1.0, size=(n, 14)).astype(np.float32)
    q[:, 3] = rng.uniform(-np.pi, np.pi, n)
    q[:, 5] = rng.uniform(-np.pi, np.pi, n)
    q[:, 4] = rng.uniform(0.0, np.pi, n)
    q[:, 6] = rng.uniform(0.0, np.pi, n)
    return np.ascontiguousarray(q)


def targets(q):
    """a smooth radiance field of the query, so that training has something to learn"""
    t = np.stack([0.5 + 0.5 * np.sin(6 * q[:, 0] + q[:, 8]), q[:, 1] * q[:, 9] + 0.1, np.abs(np.cos(4 * q[:, 2])) * q[:, 10]], 1)
    return np.ascontiguousarray(t.astype(np.float32) * 2.0)


def layer_slices(num_matrix_weights, num_params):
    s, out = 0, {}
    for l in range(HIDDEN):
        out[f"W{l}"] = slice(s, s + 64 * 64)
        s += 64 * 64
    out[f"W{HIDDEN}"] = slice(s, s + 16 * 64)
    out["grid"] = slice(num_matrix_weights, num_params)
    return out


def inputs():
    """every query / target batch of the check, drawn from one stream in a fixed order: inference, one training step, four
    training steps, inference after training"""
    rng = np.random.default_rng(23)
    q = queries(rng, N_INF)
    qt = queries(rng, N_TR)
    steps = [queries(rng, N_TR) for _ in range(4)]
    qe = queries(rng, N_INF)
    return q, (qt, targets(qt)), [(qs, targets(qs)) for qs in steps], qe


def start_params(num_params, num_matrix_weights):
    """identical, half-representable weights of working magnitude for every arm (float16)"""
    return engine.random_nrc_params(num_params, num_matrix_weights, seed=31, grid_amplitude=0.5)


def tcnn_outputs(num_matrix_weights):
    """everything the comparison reads from tiny-cuda-nn, for all rows and parameters; and the trained network (for timing)"""
    ref = TcnnNrc()
    q, (qt, tt), steps, qe = inputs()
    # init: Trainer{seed 1337}
    out = {"num_params": ref.num_params, "master_sha256": digest(ref.read(0)), "training_sha256": digest(ref.read(1)),
           "inference_all_zero": not ref.read(2).any()}
    master = start_params(ref.num_params, num_matrix_weights).astype(np.float32)
    ref.set_params(master)
    out["forward"] = ref.infer(q)
    out["loss"], out["gradients"] = ref.forward_backward(qt, tt)
    # four full training steps (forward, loss, backward, Adam, EMA) from the same start
    ref2 = TcnnNrc()
    ref2.set_params(master)
    out["losses"] = np.asarray([ref2.train(qs, ts) for qs, ts in steps], dtype=np.float32)
    out["training"], out["inference"] = ref2.read(1), ref2.read(2)
    out["after_training"] = ref2.infer(qe)
    out["rows"], out["params"] = np.arange(N_INF), np.arange(ref.num_params)
    return out, ref2


def golden_sample(out, num_matrix_weights):
    """tcnn_outputs restricted to a fixed, seeded sample of the inference rows and of each weight matrix / the hash grid"""
    rng = np.random.default_rng(7)
    rows = np.sort(rng.choice(N_INF, GOLDEN_ROWS, replace=False))
    idx = np.concatenate([sl.start + np.sort(rng.choice(sl.stop - sl.start, GOLDEN_PARAMS[name], replace=False))
                          for name, sl in layer_slices(num_matrix_weights, int(out["num_params"])).items()])
    g = {k: out[k] for k in ("num_params", "master_sha256", "training_sha256", "inference_all_zero", "loss", "losses")}
    g.update(rows=rows, params=idx, forward=out["forward"][rows], after_training=out["after_training"][rows],
             gradients=out["gradients"][idx].astype(np.float16), training=out["training"][idx], inference=out["inference"][idx])
    return g


def compare(ref, ctx):
    """this repo's network and the oracle against tiny-cuda-nn's outputs `ref` (tcnn_outputs or golden_sample): every relative
    L2 against tiny-cuda-nn is taken over ref's rows / parameters, the others over all of them"""
    rows, idx = ref["rows"], ref["params"]
    result = {}
    ours = engine.NeuralRadianceCache(ctx, HIDDEN, LR)
    assert ours.num_params == int(ref["num_params"]), (ours.num_params, int(ref["num_params"]))
    P = ours.num_params
    onet = O.OracleNrc(HIDDEN, LR)
    M = onet.num_matrix_weights
    # per weight matrix / hash grid: the slice of all parameters and the mask of ref's parameters that fall into it
    slices = {name: (sl, (idx >= sl.start) & (idx < sl.stop)) for name, sl in layer_slices(M, P).items()}
    q, (qt, tt), steps, qe = inputs()

    # ---- init: Trainer{seed 1337}
    result["init"] = {"params": int(P), "master_equal": digest(ours.read(abi.NRC_READ_MASTER)) == str(ref["master_sha256"]),
                      "training_half_equal": digest(ours.read(abi.NRC_READ_TRAINING)) == str(ref["training_sha256"]),
                      "inference_all_zero": bool(ref["inference_all_zero"]) and not ours.read(abi.NRC_READ_INFERENCE).any()}

    # ---- forward and one training step from identical weights
    params = start_params(P, M)
    master = params.astype(np.float32)
    ours.set_params(params)
    onet.set_params(params)
    dout = torch.empty((N_INF, 3), device="cuda")

    def our_infer(x):
        ours.infer(torch.from_numpy(x).cuda(), dout, N_INF)
        torch.cuda.synchronize()
        return dout.cpu().numpy()
    our_out = our_infer(q)
    o32 = onet.infer(q)
    onet.set_accumulate_half(True)
    o16 = onet.infer(q)
    onet.set_accumulate_half(False)
    ref_out = ref["forward"]
    result["forward"] = {"n": len(rows), "ours_vs_tcnn": rel_l2(our_out[rows], ref_out), "oracle_fp32acc_vs_tcnn": rel_l2(o32[rows], ref_out),
                         "oracle_halfacc_vs_tcnn": rel_l2(o16[rows], ref_out), "ours_vs_oracle_fp32acc": rel_l2(our_out, o32),
                         "tcnn_rms": float(np.sqrt(np.mean(ref_out.astype(np.float64) ** 2)))}

    ours.keep_gradients(True)
    our_loss = ours.train(torch.from_numpy(qt).cuda(), torch.from_numpy(tt).cuda(), N_TR, want_loss=True)
    our_grad = ours.read(abi.NRC_READ_GRADIENTS)
    o_loss32 = onet.train(qt, tt)
    o_grad32 = onet.get_gradients()
    onet.set_params(params)
    onet.set_accumulate_half(True)
    o_loss16 = onet.train(qt, tt)
    o_grad16 = onet.get_gradients()
    onet.set_accumulate_half(False)
    ref_grad = ref["gradients"].astype(np.float32)
    grads = {"loss": {"tcnn": float(ref["loss"]), "ours": our_loss, "oracle_fp32acc": o_loss32, "oracle_halfacc": o_loss16}}
    for name, (sl, m) in slices.items():
        r = ref_grad[m]
        grads[name] = {"ours_vs_tcnn": rel_l2(our_grad[idx[m]], r), "oracle_fp32acc_vs_tcnn": rel_l2(o_grad32[idx[m]], r),
                       "oracle_halfacc_vs_tcnn": rel_l2(o_grad16[idx[m]], r), "ours_vs_oracle_fp32acc": rel_l2(our_grad[sl], o_grad32[sl]),
                       "tcnn_norm": float(np.linalg.norm(r.astype(np.float64))), "tcnn_nonzero": int(np.count_nonzero(r)),
                       "compared": int(m.sum())}
    result["gradients"] = grads

    # ---- four full training steps (forward, loss, backward, Adam, EMA) from the same start
    ours.set_params(params)
    onet.set_params(params)
    losses = {"tcnn": [float(x) for x in ref["losses"]], "ours": [], "oracle_fp32acc": []}
    for qs, ts in steps:
        losses["ours"].append(ours.train(torch.from_numpy(qs).cuda(), torch.from_numpy(ts).cuda(), N_TR, want_loss=True))
        losses["oracle_fp32acc"].append(onet.train(qs, ts))
    weights = {"losses": losses}
    ref_tr, ref_inf = ref["training"].astype(np.float32), ref["inference"].astype(np.float32)
    our_tr = ours.read(abi.NRC_READ_TRAINING).astype(np.float32)[idx]
    our_inf = ours.read(abi.NRC_READ_INFERENCE).astype(np.float32)[idx]
    orc_tr, orc_inf = onet.get_params(ema=False).astype(np.float32)[idx], onet.get_params(ema=True).astype(np.float32)[idx]
    start = master[idx]
    delta_ref = ref_tr - start       # what four steps changed: the comparison that matters is on the update, not on the weights
    for name, (_, m) in slices.items():
        weights[name] = {"training_ours_vs_tcnn": rel_l2(our_tr[m], ref_tr[m]), "inference_ours_vs_tcnn": rel_l2(our_inf[m], ref_inf[m]),
                         "training_oracle_vs_tcnn": rel_l2(orc_tr[m], ref_tr[m]), "inference_oracle_vs_tcnn": rel_l2(orc_inf[m], ref_inf[m]),
                         "update_ours_vs_tcnn": rel_l2(our_tr[m] - start[m], delta_ref[m]),
                         "update_oracle_vs_tcnn": rel_l2(orc_tr[m] - start[m], delta_ref[m])}
    ref_after = ref["after_training"]
    weights["inference_after_training_ours_vs_tcnn"] = rel_l2(our_infer(qe)[rows], ref_after)
    weights["inference_after_training_oracle_vs_tcnn"] = rel_l2(onet.infer(qe)[rows], ref_after)
    result["weights"] = weights
    return result, ours


def timing(ref, ours):
    """the reference's own kernels and this repo's on the same GPU, same inputs"""
    n_big = 2_116_608  # pad128(1920 * 1080 + 1920 * 1080 / 48): a 1080p NRC frame's query count
    qb = queries(np.random.default_rng(29), n_big)
    _, (qt, tt), _, _ = inputs()
    t_ref_inf = ref.time_infer(qb, 3, 20)
    dqb = torch.from_numpy(qb).cuda()
    doutb = torch.empty((n_big, 3), device="cuda")
    for _ in range(3):
        ours.infer(dqb, doutb, n_big)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(20):
        ours.infer(dqb, doutb, n_big)
    e1.record()
    torch.cuda.synchronize()
    t_our_inf = e0.elapsed_time(e1) / 20
    t_ref_tr = ref.time_train(qt, tt, 3, 40)
    dqt, dtt = torch.from_numpy(qt).cuda(), torch.from_numpy(tt).cuda()
    for _ in range(3):
        ours.train(dqt, dtt, N_TR)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(40):
        ours.train(dqt, dtt, N_TR)
    e1.record()
    torch.cuda.synchronize()
    t_our_tr = e0.elapsed_time(e1) / 40
    flop_inf, flop_tr = 18432.0 * n_big, 55296.0 * N_TR
    return {"infer_queries": n_big, "tcnn_infer_ms": t_ref_inf, "ours_infer_ms": t_our_inf,
            "tcnn_infer_tflops": flop_inf / t_ref_inf / 1e9, "ours_infer_tflops": flop_inf / t_our_inf / 1e9,
            "train_samples": N_TR, "tcnn_train_step_ms": t_ref_tr, "ours_train_step_ms": t_our_tr,
            "tcnn_train_tflops": flop_tr / t_ref_tr / 1e9, "ours_train_tflops": flop_tr / t_our_tr / 1e9}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--no-timing", action="store_true")
    ap.add_argument("--golden", help="compare against the tiny-cuda-nn outputs stored in this .npz instead of running tiny-cuda-nn")
    ap.add_argument("--write-golden", help="store a sample of tiny-cuda-nn's outputs in this .npz")
    args = ap.parse_args()
    M = O.OracleNrc(HIDDEN, LR).num_matrix_weights
    if args.golden:
        ref, tcnn = dict(np.load(args.golden)), None
    else:
        ref, tcnn = tcnn_outputs(M)
        if args.write_golden:
            np.savez_compressed(args.write_golden, **golden_sample(ref, M))
    result, ours = compare(ref, engine.Context(0))
    if tcnn is not None and not args.no_timing:
        result["timing"] = timing(tcnn, ours)
    print(json.dumps(result))
    return 0


if __name__ == "__main__":
    sys.exit(main())
