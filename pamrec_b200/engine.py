"""Device engine: owns the torch-allocated pools, binds them to libpamrec_b200.so and drives one
train / score step through the C ABI.  PyTorch is used for device memory and streams only."""
import ctypes as C
import os

import numpy as np
import torch

from . import _lib as L
from . import dist as D

EMB = "sequential/embedding/"
# table -> (buffer prefix, index of its width in emb_dims = (item, cate, user))
TABLES = {
    EMB + "item_embedding": ("item", 0),
    EMB + "cate_embedding": ("cate", 1),
    EMB + "user_long_embedding": ("ulong", 2),
    EMB + "user_short_embedding": ("ushort", 2),
}
# variables that exist in the reference graph but never receive a gradient (SURVEY.md A.4): kept on the
# host so that checkpoints carry the complete variable list of base_model.py:62.  Shapes from (n_users, emb_dims).
FROZEN = {
    EMB + "user_embedding": lambda nu, d: (nu, d[2]),
    EMB + "looptimes_embedding": lambda nu, d: (10, d[1]),
    EMB + "play_lookup": lambda nu, d: (10, 40),
}
EMB_DIMS = (16, 4, 20)               # (item, cate, user) embedding widths of config/mmoe.yaml; PAMRec's only set
_TORCH_DTYPE = {L.F32: torch.float32, L.I32: torch.int32, L.F64: torch.float64, L.U8: torch.uint8}
_ESIZE = {L.F32: 4, L.I32: 4, L.F64: 8, L.U8: 1}

DEFAULT_HP = dict(learning_rate=1e-3, beta1=0.9, beta2=0.999, epsilon=1e-8, embed_l2=1e-6, layer_l2=1e-6,
                  max_grad_norm=2.0, is_clip_norm=1, fuzhu_weight=0.5, discrepancy_loss_weight=0.1,
                  loss="cross_entropy_loss", softmax_group=1)      # hparams.loss / train_num_ngs + 1 (base_model.py:195-242)

BATCH_FIELDS = (  # name, dtype, per-row shape suffix, needed for scoring
    ("item_history", np.int32, True), ("item_cate_history", np.int32, True), ("item_loop_times_history", np.float32, True),
    ("mask", np.int32, True), ("users", np.int32, False), ("items", np.int32, False), ("cates", np.int32, False),
    ("labels_satisfied", np.float32, False), ("labels_play", np.float32, False), ("plays", np.float32, False),
)
# the satisfied-only copy of the history (IT:1069-1103): read by the sibling models only (mmoe.py:199-201)
SIBLING_FIELDS = (("satisfied_item_history", np.int32, True), ("satisfied_cate_history", np.int32, True), ("satisfied_mask", np.int32, True))
MODELS = {"pamrec": L.MODEL_PAMREC, "mmoe": L.MODEL_MMOE, "ple": L.MODEL_PLE, "sharebottom": L.MODEL_SHAREBOTTOM, "sasrec": L.MODEL_SASREC}


class PamrecError(RuntimeError):
    pass


class DeviceBatch:
    """Device copies of one feed dict plus the PamrecBatch struct pointing at them."""

    def __init__(self, tensors, batch, global_batch=0):
        self.tensors = tensors
        self.batch = batch
        self.struct = L.PamrecBatch(batch=batch, global_batch=int(global_batch),
                                    **{k: C.c_void_p(v.data_ptr()) for k, v in tensors.items()})

    def nbytes(self):
        return sum(t.numel() * t.element_size() for t in self.tensors.values())


class PendingLosses:
    """The five losses of a queued step; ``result()`` waits for their device->host copy and returns them as float32[5]."""

    def __init__(self, slot):
        self._slot, self._value = slot, None

    def result(self):
        if self._value is None:
            self._slot["event"].synchronize()
            self._value = self._slot["host"].numpy().copy()
            self._slot["owner"] = None
            self._slot = None
        return self._value


class PendingHost:
    """A queued device->host copy (Engine.to_host_async)."""

    def __init__(self, slot, n):
        self._slot, self._n, self._value = slot, n, None

    def result(self):
        if self._value is None:
            self._slot["event"].synchronize()
            self._value = self._slot["host"][:self._n].numpy().copy()
            self._slot["owner"] = None
            self._slot = None
        return self._value


class PendingHistograms:
    """Histograms queued by Engine.histograms; ``result()`` waits for their device->host copy."""

    def __init__(self, slot, plan):
        self._slot, self._plan, self._value = slot, plan, None

    def result(self):
        if self._value is None:
            slot, p = self._slot, self._plan
            slot["event"].synchronize()
            stats = slot["stats"].numpy().reshape(len(p["names"]), -1)
            pairs = slot["out"].numpy().reshape(-1, 2)
            world, out = p["world"], {}
            for s, name in enumerate(p["names"]):
                st = stats[s]
                n, lo = int(st[4]), int(p["offsets"][s])
                if n > p["offsets"][s + 1] - lo:
                    raise PamrecError(f"histogram of {name}: {n} compacted entries, room for {p['offsets'][s + 1] - lo}")
                out[name] = dict(min=float(st[5:5 + world].min()), max=float(st[5 + world:5 + 2 * world].max()), num=float(st[0]),
                                 sum=float(st[1]), sum_squares=float(st[2]), nonfinite=int(st[3]),
                                 bucket_limit=pairs[lo:lo + n, 0].copy(), bucket=pairs[lo:lo + n, 1].copy())
            self._value = out
            slot["owner"] = None
            self._slot = None
        return self._value


class PendingRank:
    """Engine.rank_candidates: ``result()`` waits for the device->host copies and gives (topk_items [B,K] int32, topk_scores [B,K]
    float32, own_rank [B] int32 or None)."""

    def __init__(self, host, event, want_rank):
        self._host, self._event, self._want_rank, self._value = host, event, want_rank, None

    def result(self):
        if self._value is None:
            self._event.synchronize()
            items, scores, ranks = (t.numpy().copy() for t in self._host)
            self._value = (items, scores, ranks if self._want_rank else None)
            self._host = None
        return self._value


class PendingAttention:
    """Engine.attention: ``result()`` waits for the device->host copies and gives dict(pred [B] float32, pool [B, P, T] float32,
    maps [B, 2, T, T] float32 or None)."""

    def __init__(self, host, event):
        self._host, self._event, self._value = host, event, None

    def result(self):
        if self._value is None:
            self._event.synchronize()
            pred, pool, maps = self._host
            # the pinned buffers belong to this result alone: handed out without a further host copy
            self._value = dict(pred=pred.numpy(), pool=pool.numpy(), maps=None if maps is None else maps.numpy())
            self._host = None
        return self._value


class Engine:
    def __init__(self, n_users, n_items, n_cates, max_seq_len, max_batch, hp=None, sparse_adam="dense_exact",
                 world_size=1, rank=0, tables=None, model="pamrec", graph=None, emb_dims=EMB_DIMS):
        """model: "pamrec" (PAMRECModel) or one of the sibling baselines "mmoe" (MMoEModel_original), "ple" (PLEModel),
        "sharebottom" (ShareBottomModel), "sasrec" (SASRecModel) - those run on one GPU with whole tables.
        emb_dims: (item, cate, user) embedding widths.  PAMRec runs (16, 4, 20) only; the sibling models run (item, cate) = (16, 4)
        or (32, 8) (the reference's ple.yaml / sharebottom.yaml / sasrec.yaml) with user = 16, 20 or 40.
        graph: replay the train step from a CUDA graph (one graph per resident / staged DeviceBatch, captured at its second use;
        one GPU, whole tables, PAMRec only).  None reads PAMREC_GRAPH (default on; PAMREC_GRAPH=0 launches kernel by kernel).
        tables: "local" (whole tables on this GPU, world_size 1), "replicated" (every rank holds whole tables; the merged
        row gradients are all-reduced with the dense gradients and every rank applies the same update), "sharded" (row r on
        rank r % world_size, rows and row gradients exchanged by all-to-all; also runs on one GPU) or "auto" / None: local on one
        GPU; on several, replicated while the four tables together stay below REPLICATE_BYTES (PAMREC_REPLICATE_MB), else sharded."""
        self.lib = L.load()
        self.world, self.rank = int(world_size), int(rank)
        if model not in MODELS:
            raise PamrecError(f"unknown model {model!r}: one of {sorted(MODELS)}")
        self.model = model
        self.batch_fields = BATCH_FIELDS + (SIBLING_FIELDS if model != "pamrec" else ())
        if model != "pamrec" and (self.world != 1 or tables not in (None, "auto", "local")):
            raise PamrecError("the sibling models (mmoe / ple / sharebottom / sasrec) run on one GPU with whole tables")
        # SASRecModel has neither the user_long / user_short tables nor play_lookup (sasrec.py:20-34 on top of SBM:562-593)
        self.tables_by_name = {n: v for n, v in TABLES.items() if model != "sasrec" or v[0] in ("item", "cate")}
        try:
            limit = float(os.environ.get("PAMREC_REPLICATE_MB", D.REPLICATE_BYTES / 2 ** 20)) * 2 ** 20
            tables = D.choose_tables(tables, self.world, n_users, n_items, n_cates, limit)
        except ValueError as e:
            raise PamrecError(str(e))
        self.tables = tables
        h = dict(DEFAULT_HP)
        if hp:
            h.update(hp)
        self.hp = h
        self.dims = (int(n_users), int(n_items), int(n_cates), int(max_seq_len), int(max_batch))
        self.emb_dims = tuple(int(d) for d in emb_dims)
        mode = {"dense_exact": L.ADAM_DENSE_EXACT, "lazy": L.ADAM_LAZY}[sparse_adam]
        self.cfg = L.PamrecConfig(
            n_users=n_users, n_items=n_items, n_cates=n_cates, max_seq_len=max_seq_len, max_batch=max_batch,
            learning_rate=h["learning_rate"], beta1=h["beta1"], beta2=h["beta2"], epsilon=h["epsilon"],
            embed_l2=h["embed_l2"], layer_l2=h["layer_l2"], max_grad_norm=h["max_grad_norm"],
            is_clip_norm=int(h["is_clip_norm"]), fuzhu_weight=h["fuzhu_weight"],
            order_weight=h["discrepancy_loss_weight"], sparse_adam_mode=mode, world_size=world_size, rank=rank,
            table_mode={"local": L.TABLES_LOCAL, "sharded": L.TABLES_SHARDED, "replicated": L.TABLES_REPLICATED}[tables],
            loss_kind={"cross_entropy_loss": L.LOSS_XENT, "softmax": L.LOSS_SOFTMAX}[h["loss"]], softmax_group=int(h["softmax_group"]),
            model_kind=MODELS[model], item_dim=self.emb_dims[0], cate_dim=self.emb_dims[1], user_dim=self.emb_dims[2])
        self.handle = C.c_void_p()
        rc = self.lib.pamrec_create(C.byref(self.cfg), C.byref(self.handle))
        if rc != 0:
            raise PamrecError(f"pamrec_create failed ({rc}): check vocabulary sizes, max_seq_len <= 256, max_batch, "
                              "world_size <= 64, rank, table mode, model (siblings: one GPU, cross_entropy_loss), embedding widths "
                              f"{self.emb_dims} (item / cate / user: PAMRec 16 / 4 / 20 only; siblings 16 / 4 or 32 / 8 with user "
                              "16, 20 or 40)")
        self.dense_numel = self.lib.pamrec_dense_numel(self.handle)
        self.bn_numel = self.lib.pamrec_bn_numel(self.handle)
        self.workspace_bytes = self.lib.pamrec_workspace_bytes(self.handle)
        self.info = {p: self._query(p) for p in (L.POOL_DENSE, L.POOL_BN, L.POOL_WORKSPACE)}
        self.step = 0
        self.device = None
        if graph is None:
            graph = os.environ.get("PAMREC_GRAPH", "1") != "0"
        self.graph = bool(graph)
        self._graphs, self._profiling = {}, False
        self._dev_step = None                        # value of the device-side step counter, when known to equal self.step
        self.frozen = {n: np.zeros(f(n_users, self.emb_dims), np.float32) for n, f in FROZEN.items()
                       if model != "sasrec" or not n.endswith("play_lookup")}
        self._hist_plans, self._frozen_dev = {}, {}     # Engine.histograms: per name list, and device copies of self.frozen

    # ------------------------------------------------------------------ inventory (host only)
    def _query(self, pool):
        out = {}
        info = L.PamrecTensorInfo()
        for i in range(self.lib.pamrec_tensor_count(self.handle, pool)):
            self._check(self.lib.pamrec_tensor_info(self.handle, pool, i, C.byref(info)))
            out[info.name.decode()] = dict(offset=info.offset, numel=info.numel, dtype=info.dtype, flags=info.flags,
                                           shape=tuple(info.shape[k] for k in range(info.ndim)))
        return out

    def variable_shapes(self):
        """TF variable name -> shape for every variable of the reference graph (SURVEY.md Appendix B)."""
        nu, ni, nc, T, _ = self.dims
        shapes = {n: d["shape"] for n, d in self.info[L.POOL_DENSE].items()}
        rows = {"item": ni, "cate": nc, "ulong": nu, "ushort": nu}
        shapes.update({n: (rows[pre], self.emb_dims[k]) for n, (pre, k) in self.tables_by_name.items()})
        shapes.update({n: a.shape for n, a in self.frozen.items()})
        shapes.update({n: d["shape"] for n, d in self.info[L.POOL_BN].items()})
        return shapes

    def _check(self, rc):
        if rc != 0:
            raise PamrecError(self.lib.pamrec_last_error(self.handle).decode() or f"error {rc}")

    # ------------------------------------------------------------------ device memory
    def allocate(self, device="cuda:0"):
        if not torch.cuda.is_available():
            raise PamrecError("pamrec_b200 needs a CUDA device (sm_100a); there is no CPU path")
        self.device = torch.device(device)
        torch.cuda.set_device(self.device)
        nu, ni, nc, T, B = self.dims
        z = lambda *s: torch.zeros(*s, dtype=torch.float32, device=self.device)
        self.pool = {k: z(self.dense_numel) for k in ("dense_param", "dense_grad", "dense_m", "dense_v")}
        self.pool["bn_moving"] = z(self.bn_numel)
        di, dc, du = self.emb_dims
        for pre, rows, w in (("item", ni, di), ("cate", nc, dc), ("ulong", nu, du), ("ushort", nu, du)):
            for s in ("w", "m", "v"):
                self.pool[f"{pre}_{s}"] = z(self.table_rows(rows), w)
        self.pool["workspace"] = torch.zeros(self.workspace_bytes, dtype=torch.uint8, device=self.device)
        bufs = L.PamrecBuffers(workspace_bytes=self.workspace_bytes,
                               **{k: C.c_void_p(v.data_ptr()) for k, v in self.pool.items()})
        self._check(self.lib.pamrec_bind(self.handle, C.byref(bufs), self._stream()))
        return self

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def table_rows(self, vocab_rows):
        """Rows of this rank's buffer for a table of ``vocab_rows`` rows."""
        return int(self.lib.pamrec_shard_rows(self.handle, int(vocab_rows)))

    def init_comm(self):
        """Collective over torch.distributed's default group (any backend): rank 0 creates the NCCL unique id, everyone
        joins.  torch.distributed is the rendezvous; the step's collectives run on the library's own communicator."""
        if self.world == 1:
            return self
        import torch.distributed as dist
        from .build import nccl_library
        if not dist.is_initialized() or dist.get_world_size() != self.world or dist.get_rank() != self.rank:
            raise PamrecError("init_comm needs torch.distributed initialised with the engine's world_size / rank")
        path = nccl_library()
        cpath = path.encode() if path else None
        box = [None]
        if self.rank == 0:
            buf = C.create_string_buffer(L.COMM_ID_BYTES)
            if self.lib.pamrec_comm_unique_id(cpath, buf) != 0:
                raise PamrecError("pamrec_comm_unique_id failed (libnccl.so.2 not loadable?)")
            box[0] = buf.raw
        dist.broadcast_object_list(box, src=0)
        torch.cuda.set_device(self.device)
        self._check(self.lib.pamrec_comm_init(self.handle, cpath, box[0]))
        if self.world <= 8 and os.environ.get("PAMREC_NO_MAILBOX", "0") != "1":
            # NVLink peer mailboxes for the batch-norm sums and the gradients (kernels_head2.cu, kernels_p2p.cu): exchange the
            # cudaIpc handles
            buf = C.create_string_buffer(L.IPC_HANDLE_BYTES)
            self._check(self.lib.pamrec_comm_mailbox_create(self.handle, buf))
            handles = [None] * self.world
            dist.all_gather_object(handles, buf.raw)
            self._check(self.lib.pamrec_comm_mailbox_open(self.handle, b"".join(handles)))
            self.mailbox = True
        return self

    def all_reduce_(self, t):
        """In-place sum over ranks of a float32 / float64 / int32 device tensor on the library's communicator."""
        dt = {torch.float32: L.F32, torch.float64: L.F64, torch.int32: L.I32}[t.dtype]
        self._check(self.lib.pamrec_comm_all_reduce(self.handle, C.c_void_p(t.data_ptr()), t.numel(), dt, self._stream()))
        return t

    def _gather_table(self, shard, vocab_rows):
        """Full [vocab_rows, width] host array from every rank's shard (collective when world > 1)."""
        if self.tables != "sharded":
            return shard.detach().cpu().numpy().copy()
        if self.world == 1:
            return D.unshard_table([shard.detach().cpu().numpy()], vocab_rows)
        full = torch.zeros((self.world,) + tuple(shard.shape), dtype=shard.dtype, device=self.device)
        full[self.rank].copy_(shard)
        self.all_reduce_(full)
        return D.unshard_table(list(full.cpu().numpy()), vocab_rows)

    def dense(self, name, which="dense_param"):
        d = self.info[L.POOL_DENSE][name]
        return self.pool[which][d["offset"]:d["offset"] + d["numel"]].view(d["shape"])

    def bn(self, name):
        d = self.info[L.POOL_BN][name]
        return self.pool["bn_moving"][d["offset"]:d["offset"] + d["numel"]]

    def ws(self, name, rows=None):
        """View of a workspace tensor (first dimension optionally cut to `rows`)."""
        d = self.info[L.POOL_WORKSPACE][name]
        raw = self.pool["workspace"][d["offset"]:d["offset"] + d["numel"] * _ESIZE[d["dtype"]]]
        t = raw.view(_TORCH_DTYPE[d["dtype"]])
        shape = d["shape"]
        if rows is not None:
            inner = int(np.prod(shape[1:])) if len(shape) > 1 else 1
            return t[:rows * inner].view((rows,) + tuple(shape[1:]))
        return t.view(shape)

    # ------------------------------------------------------------------ variables by TF name
    def set_variables(self, variables):
        """variables: TF name -> array.  Unknown names raise; missing names keep their current value."""
        for name, val in variables.items():
            t = torch.as_tensor(np.asarray(val, dtype=np.float32))
            if name in self.tables_by_name:
                if self.tables == "sharded":
                    t = torch.from_numpy(D.shard_table(t.numpy(), self.world, self.rank))
                self.pool[TABLES[name][0] + "_w"].copy_(t.to(self.device))
            elif name in self.info[L.POOL_DENSE]:
                self.dense(name).copy_(t.to(self.device).view(self.dense(name).shape))
            elif name in self.info[L.POOL_BN]:
                self.bn(name).copy_(t.to(self.device))
            elif name in self.frozen:
                self.frozen[name] = np.asarray(val, dtype=np.float32).copy()
                self._frozen_dev.pop(name, None)
            else:
                raise KeyError(f"unknown variable {name}")

    def get_variables(self, pools=("var", "bn")):
        out = {}
        if "var" in pools:
            for name in self.info[L.POOL_DENSE]:
                out[name] = self.dense(name).detach().cpu().numpy().copy()
            for name, (pre, _) in self.tables_by_name.items():
                out[name] = self._gather_table(self.pool[pre + "_w"], self._vocab(pre))
            out.update({n: a.copy() for n, a in self.frozen.items()})
        if "bn" in pools:
            for name in self.info[L.POOL_BN]:
                out[name] = self.bn(name).detach().cpu().numpy().copy()
        return out

    def get_optimizer_state(self):
        st = {"step": self.step}
        for name in self.info[L.POOL_DENSE]:
            st[name + "/Adam"] = self.dense(name, "dense_m").detach().cpu().numpy().copy()
            st[name + "/Adam_1"] = self.dense(name, "dense_v").detach().cpu().numpy().copy()
        for name, (pre, _) in self.tables_by_name.items():
            st[name + "/Adam"] = self._gather_table(self.pool[pre + "_m"], self._vocab(pre))
            st[name + "/Adam_1"] = self._gather_table(self.pool[pre + "_v"], self._vocab(pre))
        return st

    def set_optimizer_state(self, st):
        """Inverse of get_optimizer_state: TF slot names (``<var>/Adam`` = m, ``<var>/Adam_1`` = v) and ``step``.  Slots that are
        missing keep their value; unknown names raise."""
        for key, val in st.items():
            if key == "step":
                self.step = int(np.asarray(val).reshape(-1)[0])
                self._dev_step = None
                continue
            name, _, slot = key.rpartition("/")
            which = {"Adam": "m", "Adam_1": "v"}.get(slot)
            if which is None:
                raise KeyError(f"unknown optimizer slot {key}")
            t = torch.as_tensor(np.asarray(val, dtype=np.float32))
            if name in self.tables_by_name:
                if self.tables == "sharded":
                    t = torch.from_numpy(D.shard_table(t.numpy(), self.world, self.rank))
                self.pool[f"{TABLES[name][0]}_{which}"].copy_(t.to(self.device))
            elif name in self.info[L.POOL_DENSE]:
                dst = self.dense(name, "dense_" + which)
                dst.copy_(t.to(self.device).view(dst.shape))
            else:
                raise KeyError(f"unknown optimizer slot {key}")

    def _vocab(self, pre):
        nu, ni, nc, _, _ = self.dims
        return {"item": ni, "cate": nc, "ulong": nu, "ushort": nu}[pre]

    # ------------------------------------------------------------------ batches
    def upload(self, feed, training=True, staged=False, global_batch=0):
        """feed: the reference's feed dict with string keys (io/sequential_iterator.py:1155-1175); with world_size > 1 it is
        this rank's share and ``global_batch`` the row count over all ranks (0 = batch * world_size).

        staged=False allocates fresh device tensors (a batch that stays resident).  staged=True packs every field into
        one pinned host buffer and issues ONE host->device copy into a reusable device buffer (two slots, alternating):
        the streaming path used by PAMRECModel.train / eval."""
        B = int(np.asarray(feed["items"]).shape[0])
        T = self.dims[3]
        need = ("item_history", "item_cate_history", "item_loop_times_history", "mask", "items", "cates") + tuple(n for n, _, _ in SIBLING_FIELDS)
        fields = []
        for name, dt, is_seq in self.batch_fields:
            if name not in feed:
                if training or name in need:
                    raise KeyError(f"feed is missing {name}")
                continue
            fields.append((name, dt, (B, T) if is_seq else (B,)))
        if B > self.dims[4]:
            raise PamrecError(f"batch {B} outside [1, {self.dims[4]}]")
        tensors = {}
        if not staged:
            for name, dt, shape in fields:
                a = np.ascontiguousarray(np.asarray(feed[name]).reshape(shape).astype(dt, copy=False))
                tensors[name] = torch.from_numpy(a).to(self.device, non_blocking=True)
            nbytes = sum(t.numel() * 4 for t in tensors.values())
        else:
            if not hasattr(self, "_stage"):
                cap = (len([f for f in self.batch_fields if f[2]]) * self.dims[4] * T + 6 * self.dims[4]) * 4 + 20 * 256
                self._stage = [dict(host=torch.empty(cap, dtype=torch.uint8).pin_memory(),
                                    dev=torch.empty(cap, dtype=torch.uint8, device=self.device),
                                    done=torch.cuda.Event()) for _ in range(2)]
                self._stage_i = 0
            slot = self._stage[self._stage_i]
            self._stage_i ^= 1
            slot["done"].synchronize()                       # the previous copy out of this pinned slot has finished
            key = (B, tuple(name for name, _, _ in fields))
            cached = slot.get("layout")
            if cached is None or cached[0] != key:
                # (re)build the views of this slot for this batch shape: host numpy views, device tensors, the C struct
                host_np = slot["host"].numpy()
                off, hv, dv = 0, [], {}
                for name, dt, shape in fields:
                    n = int(np.prod(shape)) * 4
                    hv.append((name, host_np[off:off + n].view(dt).reshape(shape)))
                    tdt = torch.int32 if dt == np.int32 else torch.float32
                    dv[name] = slot["dev"][off:off + n].view(tdt).view(shape)
                    off += (n + 255) // 256 * 256
                for name, _, _ in self.batch_fields:
                    if name not in dv:
                        dv[name] = torch.empty(0, device=self.device)
                db = DeviceBatch(dv, B, global_batch)
                for name, _, _ in self.batch_fields:
                    if dv[name].numel() == 0:
                        setattr(db.struct, name, None)
                db.h2d_bytes = off
                cached = slot["layout"] = (key, hv, db, off)
            _, hv, db, off = cached
            for name, view in hv:
                np.copyto(view, np.asarray(feed[name]).reshape(view.shape), casting="unsafe")
            slot["dev"][:off].copy_(slot["host"][:off], non_blocking=True)
            slot["done"].record(torch.cuda.current_stream(self.device))
            db.struct.global_batch = int(global_batch)
            return db
        for name, _, _ in self.batch_fields:     # scoring: unused pointers stay null
            if name not in tensors:
                tensors[name] = torch.empty(0, device=self.device)
        db = DeviceBatch(tensors, B, global_batch)
        db.h2d_bytes = nbytes
        for name, _, _ in self.batch_fields:
            if tensors[name].numel() == 0:
                setattr(db.struct, name, None)
        return db

    # ------------------------------------------------------------------ steps
    def gather(self, db):
        self._check(self.lib.pamrec_gather_fwd(self.handle, C.byref(db.struct), None, self._stream()))
        return self.ws("x0", db.batch)

    def forward(self, db, training=False, want_pred=True):
        pred = torch.empty(db.batch, dtype=torch.float32, device=self.device) if want_pred else None
        self._check(self.lib.pamrec_forward(self.handle, C.byref(db.struct), int(training),
                                            C.c_void_p(pred.data_ptr()) if want_pred else None, self._stream()))
        return pred

    def backward(self, db):
        self._check(self.lib.pamrec_backward(self.handle, C.byref(db.struct), self._stream()))

    def apply_gradients(self, db):
        self.step += 1
        self._check(self.lib.pamrec_apply_gradients(self.handle, C.byref(db.struct), self.step, self._stream()))
        self._dev_step = self.step
        return self.ws("losses")[:5]

    def train_step(self, db, losses_out=None):
        """One optimisation step; returns a device tensor [loss, data, regular, auxiliary, order] (pamrec.py:444-448)."""
        if losses_out is None and self._dev_step == self.step and self._graph_ok():
            db.graph_uses = getattr(db, "graph_uses", 0) + 1
            if db.graph_uses >= 2:                   # a batch that comes back (resident, or a staging slot): worth a capture
                return self._train_step_graph(db)
        self.step += 1
        if losses_out is None:
            losses_out = torch.empty(5, dtype=torch.float32, device=self.device)
        self._check(self.lib.pamrec_train_step(self.handle, C.byref(db.struct), self.step,
                                               C.c_void_p(losses_out.data_ptr()), self._stream()))
        self._dev_step = self.step                   # a call with step >= 1 sets the device counter
        return losses_out

    def _graph_ok(self):
        return self.graph and self.world == 1 and self.model == "pamrec" and self.tables == "local" and not self._profiling

    def _train_step_graph(self, db):
        """The step as ONE CUDA-graph launch.  The captured launches freeze their arguments, so a graph belongs to one DeviceBatch
        (its device pointers and row count) and the optimiser step lives on the device: pamrec_train_step(step = 0) makes every
        Adam kernel read lr_t from memory that a one-thread kernel at the head of the step advances (kernels_optim.cu:k_adam_step).
        The returned losses tensor is owned by the graph and overwritten by its next replay."""
        ent = self._graphs.get(id(db))
        if ent is None or ent["db"] is not db or ent["batch"] != db.batch:
            losses = torch.empty(5, dtype=torch.float32, device=self.device)
            g = torch.cuda.CUDAGraph()
            cap = torch.cuda.Stream(self.device)
            cap.wait_stream(torch.cuda.current_stream(self.device))
            with torch.cuda.graph(g, stream=cap):
                self._check(self.lib.pamrec_train_step(self.handle, C.byref(db.struct), 0, C.c_void_p(losses.data_ptr()), self._stream()))
            torch.cuda.current_stream(self.device).wait_stream(cap)
            ent = self._graphs[id(db)] = dict(graph=g, losses=losses, db=db, batch=db.batch)
        self.step += 1
        self._dev_step = self.step
        ent["graph"].replay()
        return ent["losses"]

    def train_step_async(self, db):
        """train_step whose losses travel to pinned host memory behind the step's kernels; returns a PendingLosses.  The caller
        can stage and queue the next batch while this step runs (the pipelined form of pamrec.py:440-453's blocking sess.run)."""
        if not hasattr(self, "_loss_ring"):
            self._loss_ring = [dict(host=torch.empty(5, dtype=torch.float32).pin_memory(), event=torch.cuda.Event(), owner=None)
                               for _ in range(4)]
            self._loss_i = 0
        slot = self._loss_ring[self._loss_i]
        self._loss_i = (self._loss_i + 1) % len(self._loss_ring)
        if slot["owner"] is not None:
            slot["owner"].result()                          # an unread result four steps old: read it before its slot is reused
        dev = self.train_step(db)
        slot["host"].copy_(dev, non_blocking=True)
        slot["event"].record(torch.cuda.current_stream(self.device))
        slot["owner"] = PendingLosses(slot)
        return slot["owner"]

    def to_host_async(self, dev_tensor):
        """Queue a device->host copy of a float32 device tensor into a pinned ring slot; ``.result()`` waits and returns numpy."""
        n = dev_tensor.numel()
        if not hasattr(self, "_host_ring"):
            self._host_ring, self._host_i = [], 0
        if len(self._host_ring) < 4:
            self._host_ring.append(dict(host=torch.empty(max(n, self.dims[4] * max(self.world, 1)), dtype=torch.float32).pin_memory(),
                                        event=torch.cuda.Event(), owner=None))
            slot = self._host_ring[-1]
        else:
            slot = self._host_ring[self._host_i]
            self._host_i = (self._host_i + 1) % len(self._host_ring)
            if slot["owner"] is not None:
                slot["owner"].result()
        if slot["host"].numel() < n:
            slot["host"] = torch.empty(n, dtype=torch.float32).pin_memory()
        slot["host"][:n].copy_(dev_tensor.reshape(-1), non_blocking=True)
        slot["event"].record(torch.cuda.current_stream(self.device))
        slot["owner"] = PendingHost(slot, n)
        return slot["owner"]

    def histograms(self, names):
        """Queue on the engine's stream the histograms of the variables ``names`` (TF names, as get_variables() gives them), binned
        on the device with TensorFlow's default buckets (pamrec_histograms).  Returns a PendingHistograms: ``result()`` gives
        {name: dict(min, max, num, sum, sum_squares, bucket_limit, bucket, nonfinite)}, the HistogramProto fields of
        tf.summary.histogram plus the count of non-finite values.  A table is binned over its vocabulary rows.  With world_size
        > 1 this is collective (every rank passes the same names): a sharded table is binned shard by shard and the counts summed
        over the ranks; every other variable is the same on all ranks and binned by rank 0.  Every rank receives the result."""
        names = tuple(names)
        p = self._hist_plans.get(names)
        if p is None:
            p = self._hist_plans[names] = self._hist_plan(names)
        ptrs = (C.c_void_p * len(names))(*[self._hist_ptr(n) for n in names])
        slot = p["slots"][p["next"]]
        p["next"] ^= 1
        if slot["owner"] is not None:
            slot["owner"].result()
        scratch = C.c_int64(p["scratch"].numel())
        self._check(self.lib.pamrec_histograms(self.handle, ptrs, p["counts"], len(names), int(self.world > 1), p["offsets"],
                                               C.c_void_p(p["stats"].data_ptr()), C.c_void_p(p["out"].data_ptr()),
                                               C.c_void_p(p["scratch"].data_ptr()), C.byref(scratch), self._stream()))
        slot["stats"].copy_(p["stats"], non_blocking=True)
        slot["out"].copy_(p["out"], non_blocking=True)
        slot["event"].record(torch.cuda.current_stream(self.device))
        slot["owner"] = PendingHistograms(slot, p)
        return slot["owner"]

    def _hist_plan(self, names):
        """Segment sizes, output offsets and the device / pinned buffers of one list of names (kept for the engine's lifetime)."""
        if not 1 <= len(names) <= L.HIST_MAX_SEGMENTS:
            raise PamrecError(f"histograms of 1 to {L.HIST_MAX_SEGMENTS} variables per call, not {len(names)}")
        shapes = self.variable_shapes()
        counts, caps = [], []
        for name in names:
            if name not in shapes:
                raise KeyError(f"unknown variable {name}")
            total = int(np.prod(shapes[name]))
            if name in self.tables_by_name and self.tables == "sharded":
                pre, k = self.tables_by_name[name]
                mine = len(range(self.rank, self._vocab(pre), self.world)) * self.emb_dims[k]   # this shard's vocabulary rows
            else:
                mine = total if self.rank == 0 else 0
            counts.append(mine)
            caps.append(min(L.HIST_BUCKETS, 2 * total + 1))
        offsets = np.concatenate([[0], np.cumsum(caps)]).astype(np.int64)
        counts_c = (C.c_int64 * len(names))(*counts)
        offsets_c = (C.c_int64 * (len(names) + 1))(*offsets.tolist())
        need = C.c_int64(0)
        self._check(self.lib.pamrec_histograms(self.handle, None, counts_c, len(names), int(self.world > 1), None, None, None, None,
                                               C.byref(need), None))
        sw = 5 + 2 * self.world
        f64 = lambda n, **kw: torch.empty(n, dtype=torch.float64, **kw)
        return dict(names=names, world=self.world, counts=counts_c, offsets=offsets_c, next=0,
                    scratch=torch.empty(need.value, dtype=torch.uint8, device=self.device),
                    stats=f64(len(names) * sw, device=self.device), out=f64(int(offsets[-1]) * 2, device=self.device),
                    slots=[dict(stats=f64(len(names) * sw).pin_memory(), out=f64(int(offsets[-1]) * 2).pin_memory(),
                                event=torch.cuda.Event(), owner=None) for _ in range(2)])

    def _hist_ptr(self, name):
        if name in self.tables_by_name:
            return self.pool[self.tables_by_name[name][0] + "_w"].data_ptr()
        if name in self.info[L.POOL_DENSE]:
            return self.dense(name).data_ptr()
        if name in self.info[L.POOL_BN]:
            return self.bn(name).data_ptr()
        if name not in self._frozen_dev:                         # host-side constants: one device copy until set_variables
            self._frozen_dev[name] = torch.from_numpy(self.frozen[name]).to(self.device)
        return self._frozen_dev[name].data_ptr()

    def rank_candidates(self, db, cand_items, cand_cates, top_k, exclude_history=False, want_rank=False):
        """Score every line of the scoring batch ``db`` against every candidate and keep the best ``top_k`` per line
        (pamrec_rank_candidates: score descending, then item id ascending; slots past the last candidate hold id -1, score -inf).
        cand_items / cand_cates: unique item ids in [1, n_items) and their categories (device tensors or arrays).  exclude_history
        skips the candidates at a real position of a line's history, except the line's own item.  want_rank: also the rank of each
        line's own item among the candidates (-1 when it is not one).  Overwrites the activation workspace like forward(training=False).
        Returns a PendingRank."""
        if self.world != 1 or self.tables != "local":
            raise PamrecError("rank_candidates runs on one GPU with whole tables")
        if not 1 <= int(top_k) <= L.RANK_MAX_K:
            raise PamrecError(f"top_k {top_k} outside [1, {L.RANK_MAX_K}]")
        as_dev = lambda a: torch.as_tensor(np.asarray(a.cpu() if torch.is_tensor(a) else a, np.int32)).to(self.device).contiguous()
        items, cates = as_dev(cand_items).reshape(-1), as_dev(cand_cates).reshape(-1)
        if items.numel() != cates.numel():
            raise PamrecError(f"{items.numel()} candidate items but {cates.numel()} categories")
        need = int(self.lib.pamrec_rank_scratch_bytes(self.handle, int(top_k)))
        if need < 0:
            self._check(-1)
        if getattr(self, "_rank_scratch", None) is None or self._rank_scratch.numel() < need:
            self._rank_scratch = torch.empty(need, dtype=torch.uint8, device=self.device)
        B, K = db.batch, int(top_k)
        out = (torch.empty((B, K), dtype=torch.int32, device=self.device), torch.empty((B, K), dtype=torch.float32, device=self.device),
               torch.empty(B, dtype=torch.int32, device=self.device))
        ptr = lambda t: C.c_void_p(t.data_ptr())
        self._check(self.lib.pamrec_rank_candidates(self.handle, C.byref(db.struct), ptr(items), ptr(cates), items.numel(), K,
                                                    int(bool(exclude_history)), ptr(self._rank_scratch), self._rank_scratch.numel(),
                                                    ptr(out[0]), ptr(out[1]), ptr(out[2]) if want_rank else None, self._stream()))
        host = tuple(torch.empty(t.shape, dtype=t.dtype).pin_memory() for t in out)
        for hst, dev in zip(host, out):
            hst.copy_(dev, non_blocking=True)
        event = torch.cuda.Event()
        event.record(torch.cuda.current_stream(self.device))
        return PendingRank(host, event, want_rank)

    def attention(self, db, maps=False):
        """The attention weights behind each score of the scoring batch ``db`` (pamrec_attention): the forward pass runs as in
        forward(training=False), whose predictions ``pred`` it also returns bit for bit.  ``pool`` [B, P, T]: the read-out weights
        over the history (PAMRec: its pooling weights, P = 1; MMoE / PLE / share-bottom: slot 0 the satisfied-only branch, slot 1
        the full-history branch; SASRec: block 1's attention row at the position its tower reads, P = 1).  maps=True (PAMRec and
        SASRec): also the softmax probabilities of both encoder blocks, [B, 2, T, T] (query row, key column).  One GPU with whole
        tables; overwrites the activation workspace like forward(training=False).  Returns a PendingAttention."""
        if self.world != 1 or self.tables != "local":
            raise PamrecError("attention runs on one GPU with whole tables")
        if maps and self.model not in ("pamrec", "sasrec"):
            raise PamrecError(f"attention maps: {self.model} has no self-attention encoder")
        B, T = db.batch, self.dims[3]
        P = 2 if self.model in ("mmoe", "ple", "sharebottom") else 1
        f32 = lambda *shape: torch.empty(shape, dtype=torch.float32, device=self.device)
        out = (f32(B), f32(B, P, T), f32(B, 2, T, T) if maps else None)
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        self._check(self.lib.pamrec_attention(self.handle, C.byref(db.struct), ptr(out[0]), ptr(out[1]), ptr(out[2]), self._stream()))
        host = tuple(None if t is None else torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in out)
        for hst, dev in zip(host, out):
            if dev is not None:
                hst.copy_(dev, non_blocking=True)
        event = torch.cuda.Event()
        event.record(torch.cuda.current_stream(self.device))
        return PendingAttention(host, event)

    def set_debug(self, flags):
        """Test hooks (include/pamrec_b200.h: PAMREC_DEBUG_*)."""
        self._check(self.lib.pamrec_set_debug(self.handle, int(flags)))

    def head_trace(self, backward=False):
        """ns from the start of the last persistent head kernel to each of its barrier releases and to the end of CTA 0
        (needs set_debug(DEBUG_HEAD_TRACE) before the step)."""
        buf = (C.c_uint64 * 32)()
        self._check(self.lib.pamrec_head_trace(self.handle, int(backward), buf))
        n, t0 = int(buf[29]), int(buf[31])
        return [int(buf[i]) - t0 for i in range(n)] + [int(buf[30]) - t0]

    def head_trace_ctas(self, backward=False):
        """[16, 256] ns at which every CTA of the last persistent head kernel arrived at every barrier (0 = unused)."""
        buf = (C.c_uint64 * (16 * 256))()
        self._check(self.lib.pamrec_head_trace_ctas(self.handle, int(backward), buf))
        return np.frombuffer(buf, dtype=np.uint64).reshape(16, 256).copy()

    def profile(self, on=True):
        self._profiling = bool(on)                   # per-launcher CUDA events: the step is launched kernel by kernel, not replayed
        self._check(self.lib.pamrec_profile_enable(self.handle, int(on)))
        self._check(self.lib.pamrec_profile_reset(self.handle))

    def profile_table(self):
        """{launcher: (total_ms, timed launches)}; synchronises the device first."""
        torch.cuda.synchronize(self.device)
        out = {}
        name = C.create_string_buffer(64)
        ms, n = C.c_double(), C.c_int64()
        for i in range(self.lib.pamrec_profile_count(self.handle)):
            self._check(self.lib.pamrec_profile_get(self.handle, i, name, C.byref(ms), C.byref(n)))
            out[name.value.decode()] = (ms.value, n.value)
        return out

    def launches(self):
        return int(self.lib.pamrec_last_launch_count(self.handle))

    def close(self):
        self._graphs = {}
        if self.handle:
            self.lib.pamrec_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
