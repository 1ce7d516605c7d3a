"""Tensor-level wrappers of the C ABI (one Python function per entry point of include/ncf_b200.h).

All tensors must be CUDA, contiguous, and of the dtype the header states; nothing here computes on
the host and nothing falls back to PyTorch ops.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional

import torch

from . import _lib
from ._lib import NcfAdamHyper, NcfAdamState, NcfGrads, NcfModel, check, current_stream, ptr


_ws_cache = {}
_ws_pinned = []   # buffers whose address a captured CUDA graph has baked in: never freed


def _workspace(device, nbytes: int):
    """A per-device scratch buffer for eager inference calls (grown on demand, reused across calls on
    the same stream).  A call made while a CUDA graph is being captured must not use it: the graph
    bakes the pointer in and a later, larger request would replace (free) the buffer under the graph.
    Captured calls therefore get a buffer of their own that stays alive for the process lifetime;
    anything that is captured routinely (FusedTrainStep's teacher forward) passes an explicit
    `workspace=` it owns instead."""
    if nbytes <= 0:
        return None
    if device.type == "cuda" and torch.cuda.is_current_stream_capturing():
        buf = torch.empty(nbytes, dtype=torch.uint8, device=device)
        _ws_pinned.append(buf)
        return buf
    key = (device.type, device.index)
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(nbytes, dtype=torch.uint8, device=device)
        _ws_cache[key] = buf
    return buf


def tower_widths(factor_num: int, num_layers: int):
    """[f*2^L, f*2^(L-1), ..., f] — reference src/ncf/models.py:20-26."""
    return [factor_num << (num_layers - k) for k in range(num_layers + 1)]


def tower_param_count(model_type: int, factor_num: int, num_layers: int) -> int:
    return int(_lib.load().ncf_tower_param_count(model_type, factor_num, num_layers))


def _i64(t: torch.Tensor, name: str) -> torch.Tensor:
    if t.dtype != torch.int64:
        raise _lib.NcfError(f"{name} must be int64, got {t.dtype}")
    return t


def _f32(t: torch.Tensor, name: str) -> torch.Tensor:
    if t.dtype != torch.float32:
        raise _lib.NcfError(f"{name} must be float32, got {t.dtype}")
    return t


TOWER_MATH = {"fp32": 0, "tf32": 1}


def model_struct(model_type: int, factor_num: int, num_layers: int, user_num: int, item_num: int,
                 tables, linears, predict, tower_math: str = "fp32") -> NcfModel:
    """tables = (user_gmf, item_gmf, user_mlp, item_mlp); linears = [(w, b)]*L; predict = (w, b)."""
    m = NcfModel()
    m.model_type, m.factor_num, m.num_layers = model_type, factor_num, num_layers
    m.mlp_dim = factor_num << (num_layers - 1)
    m.tower_math = TOWER_MATH[tower_math]
    m.user_num, m.item_num = user_num, item_num
    m.embed_user_gmf, m.embed_item_gmf, m.embed_user_mlp, m.embed_item_mlp = (
        ptr(_f32(t, "table")) for t in tables)
    for k, (w, b) in enumerate(linears):
        m.mlp_w[k] = ptr(_f32(w, "mlp weight"))
        m.mlp_b[k] = ptr(_f32(b, "mlp bias"))
    m.predict_w, m.predict_b = ptr(_f32(predict[0], "predict")), ptr(_f32(predict[1], "predict"))
    return m


# ---- a1 -----------------------------------------------------------------------------------------
def csr_build(pos_user: torch.Tensor, pos_item: torch.Tensor, user_num: int, validate: bool = True):
    """Sorted-column CSR of the observed pairs: (rowptr int64[U+1], col int32[P]).  `validate` reads the
    library's bad-index flag back (one host sync; building the CSR is a once-per-dataset step) and raises
    on pairs outside the table, like the reference's dok_matrix fill does (IndexError)."""
    lib = _lib.load()
    P = pos_user.numel()
    dev = pos_user.device
    rowptr = torch.empty(user_num + 1, dtype=torch.int64, device=dev)
    col = torch.empty(max(P, 1), dtype=torch.int32, device=dev)
    ws_bytes = lib.ncf_csr_workspace_bytes(P, user_num)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    bad = torch.zeros(1, dtype=torch.int32, device=dev)
    check(lib.ncf_csr_build(ptr(_i64(pos_user, "pos_user")), ptr(_i64(pos_item, "pos_item")), P,
                            user_num, ptr(rowptr), ptr(col), ptr(bad), ptr(ws), ws_bytes, current_stream()),
          "ncf_csr_build")
    if validate and int(bad.item()) != 0:
        raise _lib.NcfError(f"csr_build: a (user, item) pair lies outside the table (user_num={user_num})")
    return rowptr, col[:P]


# ---- (f) on-disk formats and preprocessing --------------------------------------------------------------
def text_parse_ints(text: torch.Tensor, K: int, exact: bool = False):
    """text: uint8 CUDA tensor holding a whole file.  Returns (values int64 [n_lines, K], status int):
    the first K integers of every non-empty line (see ncf_text_parse_ints)."""
    lib = _lib.load()
    if text.dtype != torch.uint8:
        raise _lib.NcfError("text must be a uint8 tensor")
    dev, nbytes = text.device, text.numel()
    n_lines = torch.zeros(1, dtype=torch.int64, device=dev)
    ws_bytes = int(lib.ncf_text_workspace_bytes(nbytes))
    ws = torch.empty(max(ws_bytes, 256), dtype=torch.uint8, device=dev)
    tp = ptr(text) if nbytes else None
    check(lib.ncf_text_line_starts(tp, nbytes, None, 0, ptr(n_lines), ptr(ws), ws_bytes, current_stream()),
          "ncf_text_line_starts")
    n = int(n_lines.item())                                   # one host read: sizes the outputs
    starts = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    check(lib.ncf_text_line_starts(tp, nbytes, ptr(starts), n, ptr(n_lines), ptr(ws), ws_bytes, current_stream()),
          "ncf_text_line_starts")
    out = torch.empty(n, K, dtype=torch.int64, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    check(lib.ncf_text_parse_ints(tp, nbytes, ptr(starts), n, K, int(bool(exact)), ptr(out) if n else None, ptr(status),
                                  current_stream()), "ncf_text_parse_ints")
    return out, int(status.item())


def leave_one_out_split(user: torch.Tensor, item: torch.Tensor, timestamp: torch.Tensor, user_num: int):
    """-> (train [n_train, 2], test [n_test, 2]) int64 CUDA tensors, see ncf_leave_one_out_split."""
    lib = _lib.load()
    n, dev = user.numel(), user.device
    tr_u = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    tr_i = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    te_u = torch.empty(user_num, dtype=torch.int64, device=dev)
    te_i = torch.empty(user_num, dtype=torch.int64, device=dev)
    totals = torch.zeros(2, dtype=torch.int64, device=dev)
    bad = torch.zeros(1, dtype=torch.int32, device=dev)
    ws_bytes = int(lib.ncf_split_workspace_bytes(n, user_num))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    check(lib.ncf_leave_one_out_split(ptr(_i64(user, "user")), ptr(_i64(item, "item")), ptr(_i64(timestamp, "timestamp")),
                                      n, user_num, ptr(tr_u), ptr(tr_i), ptr(te_u), ptr(te_i), ptr(totals), ptr(bad),
                                      ptr(ws), ws_bytes, current_stream()), "ncf_leave_one_out_split")
    flag = int(bad.item())
    if flag == 1:
        raise _lib.NcfError("leave_one_out_split: user id outside [0, user_num) or timestamp outside [0, 2^32)")
    if flag == 2:
        raise _lib.NcfError("leave_one_out_split: a user has more than 16384 ratings")
    n_train, n_test = (int(x) for x in totals.tolist())
    return torch.stack([tr_u[:n_train], tr_i[:n_train]], 1), torch.stack([te_u[:n_test], te_i[:n_test]], 1)


def eval_negatives(rowptr: torch.Tensor, col: torch.Tensor, test_user: torch.Tensor, num_items: int, K: int, seed: int):
    """-> (negatives int64 [n, K] ascending with -1 padding, count int32 [n]), see ncf_eval_negatives."""
    n, dev = test_user.numel(), test_user.device
    out = torch.empty(n, K, dtype=torch.int64, device=dev)
    cnt = torch.empty(n, dtype=torch.int32, device=dev)
    colp = col if col.numel() else torch.zeros(1, dtype=torch.int32, device=dev)
    check(_lib.load().ncf_eval_negatives(ptr(_i64(rowptr, "rowptr")), ptr(colp), ptr(_i64(test_user, "test_user")), n,
                                         rowptr.numel() - 1, num_items, K, seed, ptr(out), ptr(cnt), current_stream()),
          "ncf_eval_negatives")
    return out, cnt


# ---- a2 -----------------------------------------------------------------------------------------
def sample_neg(rowptr, col, pos_user, num_ng: int, item_num: int, seed: int, epoch: int,
               p_offset: int = 0, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    lib = _lib.load()
    P = pos_user.numel()
    if out is None:
        out = torch.empty(P * num_ng, dtype=torch.int64, device=pos_user.device)
    elif out.numel() < P * num_ng:
        raise _lib.NcfError("sample_neg: out too small")
    colp = col if col.numel() else torch.zeros(1, dtype=torch.int32, device=pos_user.device)
    check(lib.ncf_sample_neg(ptr(_i64(rowptr, "rowptr")), ptr(colp), ptr(_i64(pos_user, "pos_user")),
                             P, p_offset, rowptr.numel() - 1, num_ng, item_num, seed, epoch, ptr(_i64(out, "out")),
                             current_stream()), "ncf_sample_neg")
    return out


# ---- a3 -----------------------------------------------------------------------------------------
def shuffle_epoch(pos_user, pos_item, neg_item, num_ng: int, seed: int, epoch: int, q_begin: int,
                  count: int, out_user, out_item, out_label) -> None:
    lib = _lib.load()
    if min(out_user.numel(), out_item.numel(), out_label.numel()) < count:
        raise _lib.NcfError("shuffle_epoch: output buffers too small")
    check(lib.ncf_shuffle_epoch(ptr(_i64(pos_user, "pos_user")), ptr(_i64(pos_item, "pos_item")),
                                ptr(neg_item) if neg_item is not None else None, pos_user.numel(),
                                num_ng, seed, epoch, q_begin, count, ptr(_i64(out_user, "out_user")),
                                ptr(_i64(out_item, "out_item")), ptr(_f32(out_label, "out_label")),
                                current_stream()), "ncf_shuffle_epoch")


# ---- a6 -----------------------------------------------------------------------------------------
def forward_workspace_bytes(m: NcfModel, B: int) -> int:
    n = int(_lib.load().ncf_forward_workspace_bytes(C.byref(m), B))
    if n < 0:
        raise _lib.NcfError("ncf_forward_workspace_bytes: bad model")
    return n


def forward(m: NcfModel, user: torch.Tensor, item: torch.Tensor,
            out: Optional[torch.Tensor] = None, workspace: Optional[torch.Tensor] = None) -> torch.Tensor:
    """`workspace`: caller-owned scratch of at least forward_workspace_bytes(m, B) bytes (required for
    calls that end up in a CUDA graph); default = the shared per-device buffer."""
    lib = _lib.load()
    B = user.numel()
    if item.numel() != B:
        raise _lib.NcfError("forward: user and item differ in length")
    if out is None:
        out = torch.empty(B, dtype=torch.float32, device=user.device)
    ws_bytes = int(lib.ncf_forward_workspace_bytes(C.byref(m), B))
    if ws_bytes < 0:
        raise _lib.NcfError("ncf_forward_workspace_bytes: bad model")
    if workspace is not None:
        if workspace.numel() * workspace.element_size() < ws_bytes:
            raise _lib.NcfError(f"forward: workspace of {workspace.numel() * workspace.element_size()} bytes "
                                f"is smaller than the {ws_bytes} needed")
        ws = workspace
    else:
        ws = _workspace(user.device, ws_bytes)
    check(lib.ncf_forward(C.byref(m), ptr(_i64(user, "user")), ptr(_i64(item, "item")), B,
                          ptr(_f32(out, "logits")), ptr(ws) if ws is not None else None, ws_bytes,
                          current_stream()), "ncf_forward")
    return out


# ---- a7 / a8 --------------------------------------------------------------------------------------
def loss_grad(logits, label, teacher_logits, alpha: float, loss_accum: torch.Tensor,
              dlogit: Optional[torch.Tensor]) -> None:
    lib = _lib.load()
    if loss_accum.dtype != torch.float64:
        raise _lib.NcfError("loss_accum must be float64")
    check(lib.ncf_loss_grad(ptr(_f32(logits, "logits")), ptr(_f32(label, "label")),
                            ptr(teacher_logits) if teacher_logits is not None else None, alpha,
                            logits.numel(), ptr(loss_accum),
                            ptr(dlogit) if dlogit is not None else None, current_stream()),
          "ncf_loss_grad")


def loss_grad_kd(logits, label, teacher_logits, w_task: float, w_kd: float, temperature: float, kd_mode: int,
                 loss_accum: torch.Tensor, dlogit: Optional[torch.Tensor]) -> None:
    """w_task * BCE + w_kd * KD with KD = logit MSE (kd_mode 0) or T^2-scaled soft-target MSE (kd_mode 1)."""
    if loss_accum.dtype != torch.float64:
        raise _lib.NcfError("loss_accum must be float64")
    check(_lib.load().ncf_loss_grad_kd(ptr(_f32(logits, "logits")), ptr(_f32(label, "label")),
                                       ptr(teacher_logits) if teacher_logits is not None else None, w_task, w_kd,
                                       temperature, kd_mode, logits.numel(), ptr(loss_accum),
                                       ptr(dlogit) if dlogit is not None else None, current_stream()),
          "ncf_loss_grad_kd")


def feature_kd(student: NcfModel, teacher: NcfModel, g: NcfGrads, user, item, kind: int, adapter_w, adapter_b,
               weight: float, loss_accum: torch.Tensor) -> None:
    """Feature-matching term on gmf_features (kind 0) or mlp_input (kind 1): loss value + row gradients."""
    check(_lib.load().ncf_feature_kd(C.byref(student), C.byref(teacher), C.byref(g), ptr(_i64(user, "user")),
                                     ptr(_i64(item, "item")), user.numel(), kind,
                                     ptr(adapter_w) if adapter_w is not None else None,
                                     ptr(adapter_b) if adapter_b is not None else None, weight, ptr(loss_accum),
                                     current_stream()), "ncf_feature_kd")


# ---- gradient / optimiser state ---------------------------------------------------------------------
@dataclass
class GradBuffers:
    """Owner of the tensors behind an NcfGrads struct."""
    g_user_gmf: Optional[torch.Tensor]
    g_item_gmf: Optional[torch.Tensor]
    g_user_mlp: Optional[torch.Tensor]
    g_item_mlp: Optional[torch.Tensor]
    g_tower: torch.Tensor
    user_flag: torch.Tensor
    item_flag: torch.Tensor
    user_list: torch.Tensor
    item_list: torch.Tensor
    touched_count: torch.Tensor
    flat: Optional[torch.Tensor] = None  # all float gradients as one buffer (one all-reduce in DP)

    @staticmethod
    def allocate(model_type, factor_num, num_layers, user_num, item_num, capacity, device):
        f, d = factor_num, factor_num << (num_layers - 1)
        z = lambda *s, dt=torch.float32: torch.zeros(*s, dtype=dt, device=device)
        gmf, mlp = model_type != _lib.NCF_MLP, model_type != _lib.NCF_GMF
        # flat layout [user GMF | user MLP | item GMF | item MLP | tower]: the replicated part of a
        # user-partitioned data-parallel step (items + tower) is one contiguous tail -> one all-reduce
        shapes = [(user_num, f) if gmf else None, (user_num, d) if mlp else None,
                  (item_num, f) if gmf else None, (item_num, d) if mlp else None,
                  (tower_param_count(model_type, factor_num, num_layers),)]
        sizes = [0 if s is None else (s[0] * s[1] if len(s) == 2 else s[0]) for s in shapes]
        sizes = [(n + 3) // 4 * 4 for n in sizes]  # keep every piece 16-byte aligned
        flat = z(sum(sizes))
        pieces, off = [], 0
        for s, n in zip(shapes, sizes):
            numel = 0 if s is None else (s[0] * s[1] if len(s) == 2 else s[0])
            pieces.append(None if s is None else flat[off:off + numel].view(*s))
            off += n
        pieces = [pieces[0], pieces[2], pieces[1], pieces[3], pieces[4]]   # field order of the dataclass
        return GradBuffers(
            *pieces, z(user_num, dt=torch.int32), z(item_num, dt=torch.int32),
            z(min(capacity, user_num), dt=torch.int64), z(min(capacity, item_num), dt=torch.int64),
            z(4, dt=torch.int32)[:2], flat)   # + the ticket word of the step-closing kernels behind the counts

    def struct(self) -> NcfGrads:
        g = NcfGrads()
        for name in ("g_user_gmf", "g_item_gmf", "g_user_mlp", "g_item_mlp", "g_tower", "user_flag",
                     "item_flag", "user_list", "item_list", "touched_count"):
            t = getattr(self, name)
            setattr(g, name, ptr(t) if t is not None else None)
        return g


@dataclass
class AdamBuffers:
    """Owner of the tensors behind an NcfAdamState struct."""
    m_user_gmf: Optional[torch.Tensor]
    v_user_gmf: Optional[torch.Tensor]
    m_item_gmf: Optional[torch.Tensor]
    v_item_gmf: Optional[torch.Tensor]
    m_user_mlp: Optional[torch.Tensor]
    v_user_mlp: Optional[torch.Tensor]
    m_item_mlp: Optional[torch.Tensor]
    v_item_mlp: Optional[torch.Tensor]
    m_tower: torch.Tensor
    v_tower: torch.Tensor
    user_last_step: torch.Tensor
    item_last_step: torch.Tensor
    step: torch.Tensor

    @staticmethod
    def allocate(model_type, factor_num, num_layers, user_num, item_num, device):
        f, d = factor_num, factor_num << (num_layers - 1)
        z = lambda *s, dt=torch.float32: torch.zeros(*s, dtype=dt, device=device)
        gmf, mlp = model_type != _lib.NCF_MLP, model_type != _lib.NCF_GMF
        nt = tower_param_count(model_type, factor_num, num_layers)
        return AdamBuffers(
            z(user_num, f) if gmf else None, z(user_num, f) if gmf else None,
            z(item_num, f) if gmf else None, z(item_num, f) if gmf else None,
            z(user_num, d) if mlp else None, z(user_num, d) if mlp else None,
            z(item_num, d) if mlp else None, z(item_num, d) if mlp else None,
            z(nt), z(nt), z(user_num, dt=torch.int32), z(item_num, dt=torch.int32),
            z(1, dt=torch.int64))

    def struct(self) -> NcfAdamState:
        s = NcfAdamState()
        for name, _ in NcfAdamState._fields_:
            t = getattr(self, name)
            setattr(s, name, ptr(t) if t is not None else None)
        return s


def train_workspace_bytes(m: NcfModel, B: int) -> int:
    n = int(_lib.load().ncf_train_workspace_bytes(C.byref(m), B))
    if n < 0:
        raise _lib.NcfError("ncf_train_workspace_bytes: bad model or batch")
    return n


# ---- a6 + a7 + a8 + a9 ---------------------------------------------------------------------------------
def train_step_grads(m: NcfModel, g: NcfGrads, user, item, label, teacher_logits, alpha: float,
                     loss_accum: torch.Tensor, workspace: torch.Tensor,
                     logits_out: Optional[torch.Tensor] = None) -> None:
    lib = _lib.load()
    B = user.numel()
    if item.numel() != B or label.numel() != B:
        raise _lib.NcfError("train_step_grads: user/item/label differ in length")
    if loss_accum.dtype != torch.float64:
        raise _lib.NcfError("loss_accum must be float64")
    check(lib.ncf_train_step_grads(
        C.byref(m), C.byref(g), ptr(_i64(user, "user")), ptr(_i64(item, "item")),
        ptr(_f32(label, "label")), ptr(teacher_logits) if teacher_logits is not None else None,
        alpha, B, ptr(loss_accum), ptr(logits_out) if logits_out is not None else None,
        ptr(workspace), workspace.numel() * workspace.element_size(), current_stream()),
        "ncf_train_step_grads")


def wait_embedding_grads(stream: torch.cuda.Stream) -> None:
    """`stream` waits until the row gradients of the last train_step_grads call are complete (on the
    tcgen05 path: before the weight-gradient kernel) — lets a data-parallel all-reduce of the row
    gradients overlap with the rest of the step."""
    check(_lib.load().ncf_wait_embedding_grads(C.c_void_p(stream.cuda_stream)), "ncf_wait_embedding_grads")


def backward(m: NcfModel, g: NcfGrads, user, item, dlogit, workspace: torch.Tensor) -> None:
    """Backward from a caller-supplied dloss/dlogit (autograd compatibility path)."""
    check(_lib.load().ncf_backward(
        C.byref(m), C.byref(g), ptr(_i64(user, "user")), ptr(_i64(item, "item")),
        ptr(_f32(dlogit, "dlogit")), user.numel(), ptr(workspace),
        workspace.numel() * workspace.element_size(), current_stream()), "ncf_backward")


# ---- a10 ------------------------------------------------------------------------------------------------
def mark_rows(m: NcfModel, g: NcfGrads, user, item):
    """Registers the batch's distinct rows in the touched lists (SGD path; Adam uses adam_prepare)."""
    check(_lib.load().ncf_mark_rows(C.byref(m), C.byref(g), ptr(_i64(user, "user")),
                                    ptr(_i64(item, "item")), user.numel(), current_stream()),
          "ncf_mark_rows")


def adam_prepare(m: NcfModel, g: NcfGrads, s: NcfAdamState, user, item, lr, beta1=0.9, beta2=0.999,
                 eps=1e-8):
    """Registers the batch's rows and replays their pending zero-gradient Adam steps; must
    precede train_step_grads of the same batch."""
    check(_lib.load().ncf_adam_prepare(C.byref(m), C.byref(g), C.byref(s),
                                       NcfAdamHyper(lr, beta1, beta2, eps), ptr(_i64(user, "user")),
                                       ptr(_i64(item, "item")), user.numel(), current_stream()),
          "ncf_adam_prepare")


def adam_step(m: NcfModel, g: NcfGrads, s: NcfAdamState, lr, beta1=0.9, beta2=0.999, eps=1e-8):
    check(_lib.load().ncf_adam_step(C.byref(m), C.byref(g), C.byref(s),
                                    NcfAdamHyper(lr, beta1, beta2, eps), current_stream()),
          "ncf_adam_step")


def adam_step_dense(m: NcfModel, g: NcfGrads, s: NcfAdamState, lr, beta1=0.9, beta2=0.999, eps=1e-8):
    """The Adam step over every row of the tables (no touched lists, no catch-up needed afterwards)."""
    check(_lib.load().ncf_adam_step_dense(C.byref(m), C.byref(g), C.byref(s),
                                          NcfAdamHyper(lr, beta1, beta2, eps), current_stream()),
          "ncf_adam_step_dense")


PART_USERS, PART_ITEMS, PART_TOWER = 1, 2, 4


def adam_step_dense_range(m: NcfModel, g: NcfGrads, s: NcfAdamState, user_lo: int, user_hi: int, lr,
                          beta1=0.9, beta2=0.999, eps=1e-8, parts: int = 7):
    """The all-rows Adam step over user rows [user_lo, user_hi) and every item row; `parts` masks what this
    call updates (PART_USERS | PART_ITEMS | PART_TOWER)."""
    check(_lib.load().ncf_adam_step_dense_range(C.byref(m), C.byref(g), C.byref(s),
                                                NcfAdamHyper(lr, beta1, beta2, eps), int(user_lo), int(user_hi),
                                                int(parts), current_stream()), "ncf_adam_step_dense_range")


def adam_range(p: torch.Tensor, m: torch.Tensor, v: torch.Tensor, g: torch.Tensor, step: torch.Tensor,
               lr, beta1=0.9, beta2=0.999, eps=1e-8):
    """Elementwise Adam step on flat fp32 slices (optimiser sharding in data-parallel training)."""
    check(_lib.load().ncf_adam_range(ptr(p), ptr(m), ptr(v), ptr(g), p.numel(), ptr(step),
                                     NcfAdamHyper(lr, beta1, beta2, eps), current_stream()), "ncf_adam_range")


def adam_p2p(grad_ptrs, param_ptrs, m: torch.Tensor, v: torch.Tensor, lo: int, rank: int, step: torch.Tensor,
             lr, beta1=0.9, beta2=0.999, eps=1e-8, grad_scale=None):
    """Sharded Adam step with the gradient exchange inside the kernel (ncf_adam_p2p): `grad_ptrs` /
    `param_ptrs` are the device addresses of every rank's flat gradient / parameter buffer."""
    world = len(grad_ptrs)
    ga = (C.c_void_p * world)(*grad_ptrs)
    pa = (C.c_void_p * world)(*param_ptrs)
    scale = 1.0 / world if grad_scale is None else float(grad_scale)
    check(_lib.load().ncf_adam_p2p(ga, pa, ptr(m), ptr(v), lo, m.numel(), world, rank, scale, ptr(step),
                                   NcfAdamHyper(lr, beta1, beta2, eps), current_stream()), "ncf_adam_p2p")


class PeerBuffer:
    """Zero-filled device buffer in an allocation of its own (ncf_peer_alloc), so that it can be
    exported to the other ranks of the node through CUDA IPC.  `.tensor` aliases the memory."""
    _TYPESTR = {torch.float32: "<f4", torch.int64: "<i8", torch.int32: "<i4"}

    def __init__(self, numel: int, device: torch.device, dtype: torch.dtype = torch.float32):
        self.numel, self.device, self.dtype = int(numel), device, dtype
        itemsize = torch.empty(0, dtype=dtype).element_size()
        out = C.c_void_p()
        with torch.cuda.device(device):
            check(_lib.load().ncf_peer_alloc(max(self.numel, 1) * itemsize, C.byref(out)), "ncf_peer_alloc")
        self.address = out.value
        self.__cuda_array_interface__ = {"shape": (self.numel,), "typestr": self._TYPESTR[dtype],
                                         "data": (self.address, False), "version": 2, "strides": None}
        self.tensor = torch.as_tensor(self, device=device)   # keeps a reference to self
        self._peers = []

    def handle(self) -> bytes:
        buf = C.create_string_buffer(64)
        check(_lib.load().ncf_ipc_export(self.address, buf), "ncf_ipc_export")
        return buf.raw

    def open_peer(self, handle: bytes) -> int:
        """Address, valid on this rank's device, of the buffer another rank exported."""
        out = C.c_void_p()
        with torch.cuda.device(self.device):
            check(_lib.load().ncf_ipc_open(C.create_string_buffer(handle, 64), C.byref(out)), "ncf_ipc_open")
        self._peers.append(out.value)
        return out.value

    def close_peers(self):
        for a in self._peers:
            _lib.load().ncf_ipc_close(a)
        self._peers = []

    def free(self):
        """Only after every rank has closed its mapping of this buffer (barrier in between)."""
        self.close_peers()
        if self.address:
            self.tensor = None
            _lib.load().ncf_peer_free(self.address)
            self.address = None


class PeerBarrier:
    """Rank barrier over peer memory (ncf_peer_barrier): a flag array per rank, mapped by every other rank.
    Collective construction (torch.distributed must be initialised); `wait()` enqueues the barrier on the
    current stream and can be captured in a CUDA graph."""

    def __init__(self, device: torch.device):
        import torch.distributed as dist
        self.world, self.rank = dist.get_world_size(), dist.get_rank()
        self.flags = PeerBuffer(8, device, torch.int32)
        handles = [None] * self.world
        dist.all_gather_object(handles, self.flags.handle())
        self.ptrs = [self.flags.address if r == self.rank else self.flags.open_peer(handles[r]) for r in range(self.world)]
        self.epoch = torch.zeros(1, dtype=torch.int32, device=device)
        dist.barrier()

    def wait(self) -> None:
        check(_lib.load().ncf_peer_barrier(_ptr_array(self.ptrs), self.world, self.rank, ptr(self.epoch), current_stream()),
              "ncf_peer_barrier")


def adam_finish_dense(m: NcfModel, g: NcfGrads, s: NcfAdamState):
    check(_lib.load().ncf_adam_finish_dense(C.byref(m), C.byref(g), C.byref(s), current_stream()),
          "ncf_adam_finish_dense")


def adam_flush(m: NcfModel, s: NcfAdamState, lr, beta1=0.9, beta2=0.999, eps=1e-8):
    check(_lib.load().ncf_adam_flush(C.byref(m), C.byref(s), NcfAdamHyper(lr, beta1, beta2, eps),
                                     current_stream()), "ncf_adam_flush")


def sgd_step(m: NcfModel, g: NcfGrads, lr: float):
    check(_lib.load().ncf_sgd_step(C.byref(m), C.byref(g), lr, current_stream()), "ncf_sgd_step")


# ---- a11 ------------------------------------------------------------------------------------------------
def eval_rank(scores: torch.Tensor, k: int):
    """scores [n, C] -> (hit uint8[n], rank int32[n], ndcg f32[n], topk_idx int32[n, k])."""
    lib = _lib.load()
    if scores.dim() != 2:
        raise _lib.NcfError("eval_rank: scores must be [n, C]")
    n, Cc = scores.shape
    dev = scores.device
    hit = torch.empty(n, dtype=torch.uint8, device=dev)
    rank = torch.empty(n, dtype=torch.int32, device=dev)
    ndcg = torch.empty(n, dtype=torch.float32, device=dev)
    topk = torch.empty(n, k, dtype=torch.int32, device=dev)
    check(lib.ncf_eval_rank(ptr(_f32(scores, "scores")), n, Cc, k, ptr(hit), ptr(rank), ptr(ndcg),
                            ptr(topk), current_stream()), "ncf_eval_rank")
    return hit, rank, ndcg, topk


def eval_users(m: NcfModel, users: torch.Tensor, cands: torch.Tensor, k: int):
    """users [n], cands [n, C] (column 0 = held-out item) -> (hit, rank, ndcg, topk_idx, scores)."""
    lib = _lib.load()
    if cands.dim() != 2 or cands.shape[0] != users.numel():
        raise _lib.NcfError("eval_users: cands must be [n, C] with one row per user (ragged input is rejected)")
    n, Cc = cands.shape
    dev = users.device
    hit = torch.empty(n, dtype=torch.uint8, device=dev)
    rank = torch.empty(n, dtype=torch.int32, device=dev)
    ndcg = torch.empty(n, dtype=torch.float32, device=dev)
    topk = torch.empty(n, k, dtype=torch.int32, device=dev)
    scores = torch.empty(n, Cc, dtype=torch.float32, device=dev)
    ws_bytes = int(lib.ncf_eval_workspace_bytes(C.byref(m), n, Cc))
    ws = _workspace(dev, ws_bytes)
    check(lib.ncf_eval_users(C.byref(m), ptr(_i64(users, "users")), ptr(_i64(cands, "cands")), n, Cc,
                             k, ptr(hit), ptr(rank), ptr(ndcg), ptr(topk), ptr(scores), ptr(ws),
                             ws_bytes, current_stream()), "ncf_eval_users")
    return hit, rank, ndcg, topk, scores


# ---- full-catalog recommendation ------------------------------------------------------------------------
def _caller_workspace(workspace: Optional[torch.Tensor], ws_bytes: int, what: str, device):
    if workspace is None:
        return _workspace(device, ws_bytes)
    if workspace.numel() * workspace.element_size() < ws_bytes:
        raise _lib.NcfError(f"{what}: workspace of {workspace.numel() * workspace.element_size()} bytes "
                            f"is smaller than the {ws_bytes} needed")
    return workspace


def mask_items(scores: torch.Tensor, users: torch.Tensor, rowptr: torch.Tensor, col: torch.Tensor) -> torch.Tensor:
    """In place: scores[r, c] = NaN for every item c of user users[r]'s CSR row (rowptr, col of csr_build);
    rows of users outside the CSR are NaN entirely.  Returns scores."""
    if scores.dim() != 2 or scores.shape[0] != users.numel():
        raise _lib.NcfError("mask_items: scores must be [n, C] with one row per user")
    if col.dtype != torch.int32:
        raise _lib.NcfError(f"col must be int32, got {col.dtype}")
    n, Cc = scores.shape
    colp = col if col.numel() else torch.zeros(1, dtype=torch.int32, device=scores.device)
    check(_lib.load().ncf_mask_items(ptr(_f32(scores, "scores")), n, Cc, ptr(_i64(users, "users")),
                                     rowptr.numel() - 1, ptr(_i64(rowptr, "rowptr")), ptr(colp), current_stream()),
          "ncf_mask_items")
    return scores


def topk_rows(scores: torch.Tensor, k: int, target: Optional[torch.Tensor] = None,
              workspace: Optional[torch.Tensor] = None):
    """scores [n, C] (NaN = not a candidate) -> (items int64 [n, k], scores f32 [n, k], target_rank int32 [n]
    or None): the k best columns of every row, larger score first, ties to the lower column, rows with fewer
    candidates padded with -1 / NaN; target_rank = the full rank of column target[r] (-1: not a candidate)."""
    lib = _lib.load()
    if scores.dim() != 2:
        raise _lib.NcfError("topk_rows: scores must be [n, C]")
    n, Cc = scores.shape
    dev = scores.device
    ws_bytes = int(lib.ncf_topk_rows_workspace_bytes(n, Cc, k))
    if ws_bytes < 0:
        raise _lib.NcfError(f"topk_rows: k={k} outside [1, min(1024, C={Cc})]")
    ws = _caller_workspace(workspace, ws_bytes, "topk_rows", dev)
    items = torch.empty(n, k, dtype=torch.int64, device=dev)
    top = torch.empty(n, k, dtype=torch.float32, device=dev)
    rank = None
    if target is not None:
        if target.numel() != n:
            raise _lib.NcfError("topk_rows: target must hold one column per row")
        rank = torch.empty(n, dtype=torch.int32, device=dev)
    check(lib.ncf_topk_rows(ptr(_f32(scores, "scores")), n, Cc, k,
                            ptr(_i64(target, "target")) if target is not None else None, ptr(items), ptr(top),
                            ptr(rank), ptr(ws), ws_bytes, current_stream()), "ncf_topk_rows")
    return items, top, rank


def recommend_workspace_bytes(m: NcfModel, chunk_users: int, k: int) -> int:
    n = int(_lib.load().ncf_recommend_workspace_bytes(C.byref(m), chunk_users, k))
    if n < 0:
        raise _lib.NcfError(f"ncf_recommend_workspace_bytes: bad model, k={k} or chunk_users={chunk_users}")
    return n


def recommend(m: NcfModel, users: torch.Tensor, k: int, chunk_users: int, rowptr: Optional[torch.Tensor] = None,
              col: Optional[torch.Tensor] = None, target: Optional[torch.Tensor] = None,
              workspace: Optional[torch.Tensor] = None):
    """Scores users [n] against every item of the model, excludes each user's CSR row (rowptr, col of
    csr_build; None: no exclusion) and selects as topk_rows: -> (items int64 [n, k], scores f32 [n, k],
    target_rank int32 [n] or None).  `workspace`: caller-owned scratch of recommend_workspace_bytes(m,
    min(chunk_users, n), k) bytes (required for calls that end up in a CUDA graph)."""
    lib = _lib.load()
    n, dev = users.numel(), users.device
    if (rowptr is None) != (col is None):
        raise _lib.NcfError("recommend: rowptr and col go together")
    if rowptr is not None:
        if col.dtype != torch.int32:
            raise _lib.NcfError(f"col must be int32, got {col.dtype}")
        if rowptr.numel() != m.user_num + 1:
            raise _lib.NcfError(f"recommend: rowptr has {rowptr.numel()} entries, the model {m.user_num} users")
        if not col.numel():
            col = torch.zeros(1, dtype=torch.int32, device=dev)
    items = torch.empty(n, k, dtype=torch.int64, device=dev)
    top = torch.empty(n, k, dtype=torch.float32, device=dev)
    rank = None
    if target is not None:
        if target.numel() != n:
            raise _lib.NcfError("recommend: target must hold one item per user")
        rank = torch.empty(n, dtype=torch.int32, device=dev)
    if n == 0:
        return items, top, rank
    ws_bytes = recommend_workspace_bytes(m, min(int(chunk_users), n), k)
    ws = _caller_workspace(workspace, ws_bytes, "recommend", dev)
    check(lib.ncf_recommend(C.byref(m), ptr(_i64(users, "users")), n, k,
                            ptr(_i64(rowptr, "rowptr")) if rowptr is not None else None, ptr(col),
                            ptr(_i64(target, "target")) if target is not None else None, int(chunk_users),
                            ptr(items), ptr(top), ptr(rank), ptr(ws), ws.numel() * ws.element_size(),
                            current_stream()), "ncf_recommend")
    return items, top, rank


# ---- (e) row-sharded tables -------------------------------------------------------------------------------
def train_step_grads_norm(m: NcfModel, g: NcfGrads, user, item, label, B_norm: int,
                          loss_accum: torch.Tensor, workspace: torch.Tensor, teacher_logits=None,
                          alpha: float = 1.0) -> None:
    """Fused step whose loss mean runs over B_norm >= len(user) samples (a slice of a global batch)."""
    check(_lib.load().ncf_train_step_grads_norm(
        C.byref(m), C.byref(g), ptr(_i64(user, "user")), ptr(_i64(item, "item")),
        ptr(_f32(label, "label")), ptr(teacher_logits) if teacher_logits is not None else None, alpha,
        user.numel(), int(B_norm), ptr(loss_accum), None,
        ptr(workspace), workspace.numel() * workspace.element_size(), current_stream()),
        "ncf_train_step_grads_norm")


def mark_rows_side(m: NcfModel, g: NcfGrads, rows: torch.Tensor, side: int) -> None:
    check(_lib.load().ncf_mark_rows_side(C.byref(m), C.byref(g), ptr(_i64(rows, "rows")), rows.numel(),
                                         side, current_stream()), "ncf_mark_rows_side")


def adam_catchup(m: NcfModel, g: NcfGrads, s: NcfAdamState, lr, beta1=0.9, beta2=0.999, eps=1e-8):
    check(_lib.load().ncf_adam_catchup(C.byref(m), C.byref(g), C.byref(s),
                                       NcfAdamHyper(lr, beta1, beta2, eps), current_stream()),
          "ncf_adam_catchup")


def bucket_by_owner(item: torch.Tensor, world: int):
    """-> (perm int64[n], local_idx int64[n], counts int32[world]) with samples grouped by item % world."""
    n, dev = item.numel(), item.device
    perm = torch.empty(n, dtype=torch.int64, device=dev)
    local_idx = torch.empty(n, dtype=torch.int64, device=dev)
    counts = torch.empty(world, dtype=torch.int32, device=dev)
    cursor = torch.empty(world, dtype=torch.int32, device=dev)
    check(_lib.load().ncf_bucket_by_owner(ptr(_i64(item, "item")), n, world, ptr(perm), ptr(local_idx),
                                          ptr(counts), ptr(cursor), current_stream()),
          "ncf_bucket_by_owner")
    return perm, local_idx, counts


def permute(src: torch.Tensor, perm: torch.Tensor) -> torch.Tensor:
    out = torch.empty_like(src)
    fn = {torch.int64: "ncf_permute_i64", torch.float32: "ncf_permute_f32"}[src.dtype]
    check(getattr(_lib.load(), fn)(ptr(src), ptr(_i64(perm, "perm")), src.numel(), ptr(out),
                                   current_stream()), fn)
    return out


def gather_rows(table: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    out = torch.empty(idx.numel(), table.shape[1], dtype=torch.float32, device=table.device)
    check(_lib.load().ncf_gather_rows(ptr(_f32(table, "table")), ptr(_i64(idx, "idx")), idx.numel(),
                                      table.shape[1], table.shape[0], ptr(out), current_stream()),
          "ncf_gather_rows")
    return out


def scatter_add_rows(table: torch.Tensor, idx: torch.Tensor, rows: torch.Tensor) -> None:
    check(_lib.load().ncf_scatter_add_rows(ptr(_f32(table, "table")), ptr(_i64(idx, "idx")), idx.numel(),
                                           table.shape[1], table.shape[0], ptr(_f32(rows, "rows")),
                                           current_stream()), "ncf_scatter_add_rows")


def _ptr_array(addresses):
    return (C.c_void_p * len(addresses))(*addresses)


def shard_request(item: torch.Tensor, world: int, rank: int, cap: int, item_num: int, inbox_ptrs, count_ptrs,
                  cursor: torch.Tensor) -> None:
    check(_lib.load().ncf_shard_request(ptr(_i64(item, "item")) if item.numel() else None, item.numel(), world, rank,
                                        cap, item_num, _ptr_array(inbox_ptrs), _ptr_array(count_ptrs), ptr(cursor),
                                        current_stream()), "ncf_shard_request")


def shard_mark_requests(m: NcfModel, g: NcfGrads, inbox: torch.Tensor, inbox_count: torch.Tensor, world: int,
                        cap: int) -> None:
    check(_lib.load().ncf_shard_mark_requests(C.byref(m), C.byref(g), ptr(inbox), ptr(inbox_count), world, cap,
                                              current_stream()), "ncf_shard_mark_requests")


def shard_push_rows(m: NcfModel, inbox: torch.Tensor, inbox_count: torch.Tensor, world: int, cap: int,
                    rows_gmf_ptrs, rows_mlp_ptrs) -> None:
    check(_lib.load().ncf_shard_push_rows(C.byref(m), ptr(inbox), ptr(inbox_count), world, cap,
                                          _ptr_array(rows_gmf_ptrs) if rows_gmf_ptrs else None,
                                          _ptr_array(rows_mlp_ptrs) if rows_mlp_ptrs else None, current_stream()),
          "ncf_shard_push_rows")


def shard_push_grads(item: torch.Tensor, world: int, item_num: int, g_gmf, g_mlp, f: int, d: int, grad_gmf_ptrs,
                     grad_mlp_ptrs) -> None:
    check(_lib.load().ncf_shard_push_grads(ptr(_i64(item, "item")) if item.numel() else None, item.numel(), world,
                                           item_num, ptr(g_gmf) if g_gmf is not None else None,
                                           ptr(g_mlp) if g_mlp is not None else None, f, d,
                                           _ptr_array(grad_gmf_ptrs) if grad_gmf_ptrs else None,
                                           _ptr_array(grad_mlp_ptrs) if grad_mlp_ptrs else None, current_stream()),
          "ncf_shard_push_grads")
