"""Mirror of the reference's model.py (inference side): `ResidualCNN().load_weights(path)` then
`.predict(x)` -> (p[294] float64 soft-maxed, v) exactly like Model.predict (model.py:21-24), plus
`predict_batch` for (B,7,7,7) inputs.  The arithmetic runs in libccx.so's CUDA kernels; there is no CPU path.

Weights: Keras `save_weights` HDF5 files (good_model.h5 ...) are read with h5lite (no h5py needed);
`.npz` files holding the same '<layer>/<param>' arrays are accepted too.  BatchNormalization
(eps 1e-3, Keras default) is folded into the preceding conv at load time."""
import ctypes

import numpy as np
import torch

from . import _lib, h5lite
from .config import DTYPE_BF16, DTYPE_F32, DTYPE_U8, INPUT_DIM, NUM_ACTIONS, NUM_FILTERS

BN_EPS = 1e-3


def read_weight_file(path):
    if str(path).endswith(".npz"):
        return {k: np.asarray(v, dtype=np.float32) for k, v in np.load(path).items()}
    return h5lite.read_weights(path)


def _fold(w, i):
    """conv2d_i + batch_normalization_i -> (K x Cout matrix, bias), float64 folding then float32."""
    k = w["conv2d_%d/kernel" % i].astype(np.float64)
    b = w["conv2d_%d/bias" % i].astype(np.float64)
    g, be = w["batch_normalization_%d/gamma" % i].astype(np.float64), w["batch_normalization_%d/beta" % i].astype(np.float64)
    mu, var = (w["batch_normalization_%d/moving_mean" % i].astype(np.float64),
               w["batch_normalization_%d/moving_variance" % i].astype(np.float64))
    s = g / np.sqrt(var + BN_EPS)
    kh, kw, cin, cout = k.shape
    return (k * s).reshape(kh * kw * cin, cout), (b - mu) * s + be


def pack_weights(w):
    """Keras tensors -> the flat fp32 blob ccx_net_load expects (layout: csrc/ccx_net.cu header)."""
    parts = []

    def add(i):
        m, b = _fold(w, i)
        parts.extend([m.ravel(), b.ravel()])
    add(1)                                     # model.py:62
    for blk in range(9):                       # model.py:66-76
        add(2 + 3 * blk); add(3 + 3 * blk); add(4 + 3 * blk)
    add(29)                                    # policy conv, model.py:108
    parts.extend([w["policy_head/kernel"].ravel(), w["policy_head/bias"].ravel()])
    add(30)                                    # value conv, model.py:91
    parts.extend([w["dense_1/kernel"].ravel(), w["dense_1/bias"].ravel(),
                  w["value_head/kernel"].ravel(), w["value_head/bias"].ravel()])
    return np.ascontiguousarray(np.concatenate([np.asarray(p, dtype=np.float64) for p in parts]).astype(np.float32))


def _op_layout(Wt, fp16=False):
    """[N][K] float matrix -> bf16 bytes in the UMMA K-major core-matrix operand layout (csrc/ccx_umma.cuh):
    byte offset of (n, k) = (n//8)*(K//8)*128 + (k//8)*128 + (n%8)*16 + (k%8)*2."""
    N, K = Wt.shape
    assert N % 8 == 0 and K % 8 == 0
    bits = torch.from_numpy(np.ascontiguousarray(Wt, dtype=np.float32)).to(torch.float16 if fp16 else torch.bfloat16).view(torch.int16).numpy()
    out = np.zeros(N * K, dtype=np.int16)
    n, k = np.meshgrid(np.arange(N), np.arange(K), indexing="ij")
    off = (n // 8) * (K // 8) * 64 + (k // 8) * 64 + (n % 8) * 8 + (k % 8)        # in 2-byte elements
    out[off.ravel()] = bits.ravel()
    return out


def _with_bias_columns(Wt, bias, fp16):
    """[N][K] -> [N][K + 16]: columns K, K+1 = the bias split into two 16-bit terms (hi = round16(b), lo = round16(b - hi)),
    multiplied inside the kernel by a constant ones operand (csrc/ccx_net_tc.cu, bias MMA)."""
    dt = torch.float16 if fp16 else torch.bfloat16
    b = torch.from_numpy(np.asarray(bias, dtype=np.float64))
    hi = b.to(torch.float32).to(dt).to(torch.float64)
    lo = (b - hi).to(torch.float32).to(dt).to(torch.float64)
    ext = np.zeros((Wt.shape[0], Wt.shape[1] + 16), dtype=np.float64)
    ext[:, :Wt.shape[1]] = Wt
    ext[:, Wt.shape[1]] = hi.numpy()
    ext[:, Wt.shape[1] + 1] = lo.numpy()
    return ext


def pack_weights_tc(w, fp16=False):
    """Keras tensors -> (16-bit operand blob as int16 array, fp32 blob) for ccx_net_load_tc (layout: csrc/ccx_net_tc.cu
    header).  Every weight matrix is stored transposed ([N][K + 16], bias columns appended) and BN-folded."""
    ops, fl = [], []

    def folded(i):
        m, b = _fold(w, i)                       # (K, N), (N,)
        return m, b
    m, b = folded(1)                             # conv1: K 63 -> 64
    ops.append(_op_layout(_with_bias_columns(np.pad(m, ((0, 1), (0, 0))).T, b, fp16), fp16)); fl.append(b)
    mp, bp = folded(29)                          # policy conv (64,16)
    mv, bv = folded(30)                          # value conv (64,1)
    heads = np.zeros((64, 32)); heads[:, :16] = mp; heads[:, 16] = mv[:, 0]
    hb = np.zeros(32); hb[:16] = bp; hb[16] = bv[0]
    ops.append(_op_layout(_with_bias_columns(heads.T, hb, fp16), fp16)); fl.append(hb)
    for blk in range(9):
        for i in (2 + 3 * blk, 3 + 3 * blk, 4 + 3 * blk):
            m, b = folded(i)
            ops.append(_op_layout(_with_bias_columns(m.T, b, fp16), fp16)); fl.append(b)
    Wd = np.zeros((400, 320)); Wd[:, :294] = w["policy_head/kernel"]
    bd = np.zeros(320); bd[:294] = w["policy_head/bias"]
    for half in range(2):
        Wh = Wd[:, half * 160:(half + 1) * 160]
        ops.append(_op_layout(Wh[:208].T, fp16)); ops.append(_op_layout(Wh[208:].T, fp16))
    fl.extend([bd, w["dense_1/kernel"].ravel(), w["dense_1/bias"].ravel(), w["value_head/kernel"].ravel(),
               w["value_head/bias"].ravel()])
    blob = np.ascontiguousarray(np.concatenate(ops))
    floats = np.ascontiguousarray(np.concatenate([np.asarray(f, dtype=np.float64).ravel() for f in fl]).astype(np.float32))
    return blob, floats


def pack_weights_acc(w):
    """Keras tensors -> operand blob of the accurate tensor-core mode (csrc/ccx_net_tc.cu, namespace acl): every BN-folded
    matrix as [hi: N x (K+16) with the bias columns][lo: N x K], hi = round_half(W), lo = round_half(W - hi)."""
    ops = []

    def split(Wt, bias):
        Wt = np.asarray(Wt, dtype=np.float64)
        hi = torch.from_numpy(Wt).to(torch.float32).to(torch.float16).to(torch.float64).numpy()
        lo = Wt - hi
        ops.append(_op_layout(_with_bias_columns(hi, bias, True), True))
        ops.append(_op_layout(lo, True))
    m, b = _fold(w, 1)
    split(np.pad(m, ((0, 1), (0, 0))).T, b)
    mp, bp = _fold(w, 29)
    mv, bv = _fold(w, 30)
    heads = np.zeros((64, 32)); heads[:, :16] = mp; heads[:, 16] = mv[:, 0]
    hb = np.zeros(32); hb[:16] = bp; hb[16] = bv[0]
    split(heads.T, hb)
    for blk in range(9):
        for j, i in enumerate((2 + 3 * blk, 3 + 3 * blk, 4 + 3 * blk)):
            m, b = _fold(w, i)
            if j != 1:
                split(m.T, b)
                continue
            # conv B: one [64 x (288 + 16)] operand, rows 0-31 = hi with the bias columns, rows 32-63 = lo (no bias)
            Wt = np.asarray(m.T, dtype=np.float64)
            hi = torch.from_numpy(Wt).to(torch.float32).to(torch.float16).to(torch.float64).numpy()
            both = np.concatenate([_with_bias_columns(hi, b, True), _with_bias_columns(Wt - hi, np.zeros_like(b), True)], axis=0)
            ops.append(_op_layout(both, True))
    # policy dense (400 -> 294, padded to 320): 2 N-halves x 4 K-chunks (112, 96, 96, 96) x [hi (N160, Kc) | lo (N160, Kc)]
    Wd = np.zeros((400, 320)); Wd[:, :294] = np.asarray(w["policy_head/kernel"], dtype=np.float64)
    for half in range(2):
        Wh = Wd[:, half * 160:(half + 1) * 160]
        for k0, kc in ((0, 112), (112, 96), (208, 96), (304, 96)):
            Wt = Wh[k0:k0 + kc].T
            hi = torch.from_numpy(np.ascontiguousarray(Wt)).to(torch.float32).to(torch.float16).to(torch.float64).numpy()
            ops.append(_op_layout(hi, True))
            ops.append(_op_layout(Wt - hi, True))
    return np.ascontiguousarray(np.concatenate(ops))


class Model:
    """model.py:15-47"""

    def __init__(self, input_dim, filters, version=0):
        self.input_dim, self.filters, self.version = input_dim, filters, version


class ResidualCNN(Model):
    """model.py:52-145 (inference).  `engine` is an engine.Engine; one is created on cuda:0 if omitted."""

    def __init__(self, input_dim=INPUT_DIM, filters=NUM_FILTERS, engine=None):
        Model.__init__(self, input_dim, filters)
        from .engine import Engine
        self.eng = engine or Engine()
        self.loaded = False
        self.fused_mcts = True      # engine.BatchedMCTS.search_net / BatchedSelfPlay may run the rounds inside libccx (ccx_mcts_run_net)
        # default = the accurate tensor-core mode: meets the <= 1e-3 output bar against the restated Keras graph (max |dp| 2e-5)
        # at 21.4 M self-play sims/s; set_kernel("tc") trades that for 1.7x the speed (max |dp| 3.2e-3, same argmax)
        self.kernel = "tc_acc"
        self.tc_dtype = "fp16"      # IEEE-half operands: 8x smaller error than bf16 at the same speed (see DESIGN.md §3)
        self.symmetry, self.symmetry_seed = "off", 0     # set_symmetry

    def load_weights(self, filepath):
        weights = read_weight_file(filepath)
        packed = pack_weights(weights)
        if packed.size != self.eng.L.ccx_net_num_weights():
            raise _lib.CcxError("weight file does not describe the 9-block ResidualCNN")
        self.eng.call("ccx_net_load", ctypes.c_void_p(packed.ctypes.data), packed.size)
        self._weights = weights
        self._load_tc()
        self.loaded = True
        self.set_kernel(self.kernel)
        return self

    def _load_acc(self):
        blob = pack_weights_acc(self._weights)
        assert blob.nbytes == self.eng.L.ccx_net_acc_blob_bytes()
        self.eng.call("ccx_net_load_acc", ctypes.c_void_p(blob.ctypes.data), blob.nbytes)
        self._acc_loaded = True

    def _load_tc(self):
        blob, floats = pack_weights_tc(self._weights, fp16=self.tc_dtype == "fp16")
        assert blob.nbytes == self.eng.L.ccx_net_tc_blob_bytes() and floats.size == self.eng.L.ccx_net_tc_num_floats()
        self.eng.call("ccx_net_load_tc", ctypes.c_void_p(blob.ctypes.data), blob.nbytes, ctypes.c_void_p(floats.ctypes.data),
                      floats.size, 1 if self.tc_dtype == "fp16" else 0)

    def set_kernel(self, kernel, tc_dtype=None):
        """'tc' = tcgen05 tensor-core kernels (default; operands bf16 or fp16, fp32 accumulation), 'tc_acc' = the same in split
        precision (hi + lo halves of activations and weights: fp32-level accuracy at ~1/3 of the speed), 'simt' = fp32 SIMT kernel."""
        assert kernel in ("tc", "simt", "tc_acc")
        self.kernel = kernel
        if tc_dtype is not None and tc_dtype != self.tc_dtype:
            assert tc_dtype in ("bf16", "fp16")
            self.tc_dtype = tc_dtype
            if self.loaded:
                self._load_tc()
        if self.loaded:
            if kernel == "tc_acc" and not getattr(self, "_acc_loaded", False):
                self._load_acc()
            self.eng.call("ccx_net_set_mode", {"simt": 0, "tc": 1, "tc_acc": 2}[kernel])
        return self

    SYMMETRY_MODES = {"off": 0, "random": 1, "mean": 2}

    def set_symmetry(self, mode="off", seed=0):
        """Mirror-symmetric net evaluation (ccx_net_set_symmetry), for every search that evaluates with this model's engine:
        evaluate_states, BatchedMCTS.search_net, BatchedSelfPlay, BatchedArena, the MCTS facade.  The game is symmetric under the
        mirror cell (r, c) -> (6 - c, 6 - r).  'random' evaluates each position in one orientation drawn from (seed, position),
        at no extra cost; 'mean' averages the policy and value of both orientations, at twice the net batch; 'off' (the default)
        evaluates as is.  Raw forward / predict_batch stay un-symmetrised."""
        if mode not in self.SYMMETRY_MODES:
            raise ValueError("symmetry mode must be one of %s" % sorted(self.SYMMETRY_MODES))
        self.eng.call("ccx_net_set_symmetry", self.SYMMETRY_MODES[mode], int(seed) & 0xFFFFFFFFFFFFFFFF)
        self.symmetry, self.symmetry_seed = mode, int(seed)
        return self

    # -- batched inference ---------------------------------------------------------------------------
    def forward(self, planes):
        """planes: (B,7,7,7) torch tensor on the engine's device, dtype uint8 / bfloat16 / float32.
        Returns (logits float32 (B,294), value float32 (B,))."""
        dt = {torch.uint8: DTYPE_U8, torch.bfloat16: DTYPE_BF16, torch.float32: DTYPE_F32}[planes.dtype]
        planes = planes.contiguous()
        n = planes.shape[0]
        logits = self.eng.empty((n, NUM_ACTIONS), torch.float32)
        value = self.eng.empty((n,), torch.float32)
        if self.kernel in ("tc", "tc_acc"):
            if planes.dtype != torch.uint8:
                planes = planes.to(torch.uint8)          # plane values are the integers 0..6 (utils.py:123-128)
            self.eng.call("ccx_net_forward_tc" if self.kernel == "tc" else "ccx_net_forward_u8", n, ctypes.c_void_p(planes.data_ptr()),
                          ctypes.c_void_p(logits.data_ptr()), ctypes.c_void_p(value.data_ptr()))
            return logits, value
        self.eng.call("ccx_net_forward", n, ctypes.c_void_p(planes.data_ptr()), dt,
                      ctypes.c_void_p(logits.data_ptr()), ctypes.c_void_p(value.data_ptr()))
        return logits, value

    def predict_batch(self, planes):
        """Model.predict for a batch: (p float64 (B,294) soft-maxed over all logits, v float64 (B,))."""
        logits, value = self.forward(planes)
        n = logits.shape[0]
        p = self.eng.empty((n, NUM_ACTIONS), torch.float64)
        v = self.eng.empty((n,), torch.float64)
        self.eng.call("ccx_softmax_f64", n, ctypes.c_void_p(logits.data_ptr()), ctypes.c_void_p(value.data_ptr()),
                      ctypes.c_void_p(p.data_ptr()), ctypes.c_void_p(v.data_ptr()))
        return p, v

    def predict(self, input_board):
        """model.py:21-24 — one (7,7,7) array in, (p[294], v) numpy out."""
        x = torch.from_numpy(np.ascontiguousarray(np.asarray(input_board, dtype=np.float32))[None]).to(self.eng.device)
        p, v = self.predict_batch(x)
        return p[0].cpu().numpy(), v[0].cpu().numpy()

    def evaluate_states(self, leaf_state):
        """to_model_input + predict for packed states (5+, n) int64 on the device (MCTS.py:93)."""
        n = leaf_state.shape[1]
        p = self.eng.empty((n, NUM_ACTIONS), torch.float64)
        v = self.eng.empty((n,), torch.float64)
        self.eng.call("ccx_net_eval", n, ctypes.c_void_p(leaf_state.data_ptr()), ctypes.c_void_p(p.data_ptr()),
                      ctypes.c_void_p(v.data_ptr()))
        return p, v
