"""Host-side mirror of the reference's ``SequentialIterator`` (IT = reco_utils/recommender/deeprec/io/
sequential_iterator.py in the reference tree): same text formats, same batching algorithm, same Python
``random`` call order, so batches are bit-identical to the reference's feed dicts — but the yielded
mapping is keyed by strings (the placeholder names of IT:120-163) and there is no TensorFlow.

Differences in HOW, not WHAT: a file is tokenised once into flat columns and the batching itself - the per-user
history state machine of the training branch, the listwise groups, padding, masks, play-ratio buckets and the
satisfied-only compaction - runs in native code (``csrc/batcher.cu``, host only, ``pamrec_batcher_*`` in
include/pamrec_b200.h).  Python keeps the file parsing and every ``random`` call, in the reference's order.  The
pure-Python batcher below is the same algorithm written out; it is used when noise injection is on (it draws from
``np.random`` per element), when a file has ragged history columns, or with ``PAMREC_PY_ITERATOR=1``, and the tests
hold the two implementations bit-identical.
"""
import ctypes as C
import os
import random

import numpy as np

from .deeprec_utils import load_dict

__all__ = ["SequentialIterator", "LocalFeed", "lisan", "bar_border_list", "takatak_bar_border_list_dict"]

# decile borders of play_time / duration (IT:24-42)
bar_border_list = [0.00000000e+00, 4.09545455e-02, 1.28786778e-01, 3.27894289e-01,
                   7.66666667e-01, 1.05850847e+00, 1.18596610e+00, 1.53888889e+00,
                   2.13000000e+00, 3.18951300e+03]
takatak_bar_border_list_dict = {
    10: [0.00000000e+00, 9.42727958e-02, 1.83767085e-01, 3.43377108e-01,
         5.84957075e-01, 8.40688722e-01, 1.01619134e+00, 1.06384801e+00,
         1.12731802e+00, 1.53233455e+00, 1.42410704e+02],
    8: [0., 0.11222045, 0.25718205, 0.5326864, 0.85086416,
        1.03270076, 1.08606422, 1.32310015, 34.54434426],
    6: [0., 0.14884331, 0.42646411, 0.85086416, 1.0506716,
        1.17514919, 34.54434426],
}

FEED_KEYS = (
    "labels_satisfied", "labels_play", "plays", "users", "items", "cates", "durations", "item_history",
    "item_cate_history", "item_duration_history", "mask", "item_satisfied_value_history", "item_play_value_history",
    "item_loop_times_history", "satisfied_item_history", "satisfied_cate_history", "satisfied_duration_history",
    "satisfied_play_history", "satisfied_mask")


def _borders(dataset, num):
    if dataset == "takatak":
        return takatak_bar_border_list_dict[num]
    if dataset == "wechat":
        return bar_border_list
    raise Exception("the dataset is wrong")


def lisan(x, dataset, num=10):
    """IT:43-53: max(bisect_right(borders, x) - 1, 0)."""
    return int(lisan_array(np.asarray([x]), dataset, num)[0])


def lisan_array(x, dataset, num=10):
    """Vectorised lisan; NaN sorts last exactly like bisect's `x < a[mid]` walk."""
    idx = np.searchsorted(np.asarray(_borders(dataset, num)), x, side="right") - 1
    return np.maximum(idx, 0)


def _ratio64(play, dur):
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.asarray(play, np.float64) / np.asarray(dur, np.float64)


class LocalFeed(dict):
    """One rank's share of a global batch (same 19 keys).  ``global_rows`` = rows of the whole batch; ``global_users`` [rows] /
    ``global_labels_satisfied`` [rows, 1] = those two columns for every row of it (what the scoring loops return per row)."""
    global_rows = 0
    world = 1
    rank = 0
    global_users = None
    global_labels_satisfied = None


class SequentialIterator:
    """``SequentialIterator(hparams, graph)`` — ``graph`` is accepted and ignored (IT:56)."""

    VALID_THRESHOLD = 8          # seconds, IT:96
    BEGIN_HISTORY_LEN_MAX = 5    # IT:98
    MAX_SEQUENCE = 100           # IT:476

    def __init__(self, hparams, graph=None, col_spliter="\t"):
        self.noise_train_hist = hparams.noise_train_hist
        self.noise_train_listwise = hparams.noise_train_listwise
        self.noise_only_predict = hparams.noise_only_predict
        self.dataset = hparams.dataset
        self.bucket_num = hparams.bucket_num
        _borders(self.dataset, self.bucket_num) if self.dataset in ("wechat", "takatak") else None
        dirs, _ = os.path.split(hparams.item_vocab)
        if self.dataset == "wechat":
            meta_path = os.path.join(dirs, "wechat_business_recommenders.csv")
        elif self.dataset == "takatak":
            meta_path = os.path.join(dirs, "takatak_business_recommenders.csv")
        else:
            raise Exception("there is no the dataset")
        self.meta_dict = {}                      # IT:79-86: loaded, unused by the live path
        with open(meta_path, "r") as f:
            for line in f:
                parts = line.strip().split("\t")
                iid = int(parts[0])
                if iid not in self.meta_dict:
                    self.meta_dict[iid] = [int(parts[1]), float(parts[2])]
        self.train = False
        self.shard = None                        # (world, rank) under data parallelism, see load_data_from_file
        self.col_spliter = col_spliter
        self.userdict = load_dict(hparams.user_vocab)
        self.itemdict = load_dict(hparams.item_vocab)
        self.catedict = load_dict(hparams.cate_vocab)
        self.max_seq_length = hparams.max_seq_length
        self.batch_size = hparams.batch_size
        self.iter_data = dict()
        self.time_unit = hparams.time_unit
        self.graph = graph

    # ------------------------------------------------------------------ parsing (IT:175-322)
    def _history_columns(self, words, first):
        items = [self.itemdict.get(w, 0) for w in words[first].strip().split(",")]
        cates = [self.catedict.get(w, 0) for w in words[first + 1].strip().split(",")]
        durs = [float(w) for w in words[first + 2].strip().split(",")]
        sats = [float(w) for w in words[first + 3].strip().split(",")]
        plays_ms = words[first + 4].strip().split(",")
        if self.noise_only_predict != 0:         # IT:317-318 (zip with durations bounds the length)
            plays = np.array([max(float(w) / 1000 + np.random.normal(0, self.noise_only_predict), 0)
                              for w, _ in zip(plays_ms, durs)])
        else:
            plays = np.array([float(w) / 1000 for w in plays_ms])
        durs = durs[:len(plays_ms)]              # IT:313 zips plays with durations
        return items, cates, sats, plays, durs

    def parser_one_line(self, line):
        """Train line (6 columns, one per user) or eval line (11 columns, one per impression)."""
        words = line.strip().split(self.col_spliter)
        if self.train:
            user_id = self.userdict.get(words[0], 0)
            items, cates, sats, plays, durs = self._history_columns(words, 1)
            return (user_id, items, cates, durs, sats, plays)
        label_satisfied = int(words[0])
        label_play = float(words[1]) / 1000
        user_id = self.userdict.get(words[2], 0)
        item_id = self.itemdict.get(words[3], 0)
        item_cate = self.catedict.get(words[4], 0)
        duration = float(words[5])
        items, cates, sats, plays, durs = self._history_columns(words, 6)
        return (label_satisfied, label_play, user_id, item_id, item_cate, duration, items, cates, durs, sats, plays)

    def parse_file(self, input_file):
        with open(input_file, "r") as f:
            lines = f.readlines()
        return [self.parser_one_line(line) for line in lines if line]

    # ------------------------------------------------------------------ batches
    def _lines(self, infile):
        """The file parsed by the Python parser, once (IT:366-370 caches per file the same way)."""
        if infile not in self.iter_data:
            self.iter_data[infile] = self.parse_file(infile)
        return self.iter_data[infile]

    def load_data_from_file(self, infile, batch_num_ngs=0, min_seq_length=1):
        """Generator of feed mappings (IT:334-763).  The mode switch is on the file's basename (IT:361-364)."""
        train = os.path.basename(infile) == "train_data"
        self.train = train                       # read by parser_one_line; everything below uses the local flag, so a scoring
        native = self._native(infile, train)     # pass may start on this iterator while a training generator is suspended
        # data parallel (set by the model under torch.distributed): materialise this rank's share only.  Negatives are drawn
        # from the whole batch's targets, so that path keeps global feeds (the model splits them).
        shard = self.shard if (native and batch_num_ngs == 0 and self.shard and self.shard[0] > 1) else None
        if train:
            gen = self._train_batches_native(native, shard) if native else self._train_batches(self._lines(infile))
        else:
            gen = self._eval_batches_native(native, min_seq_length, shard) if native else self._eval_batches(self._lines(infile), min_seq_length)
        if batch_num_ngs > 0:
            if not train:
                # evaluation files carry their negatives as extra lines after each positive (QS:483,493)
                raise NotImplementedError("batch_num_ngs > 0 applies to the training file only")
            gen = (self._with_negatives(b, batch_num_ngs) for b in gen)
        yield from gen

    def _with_negatives(self, res, ngs):
        """In-batch negative sampling as SPECIFIED by the reference's disabled block (IT:801-1007; the live code there is
        `exit(-1)`, so there is no executable behaviour to match - this follows the commented statements literally):
        every row is followed by `ngs` negatives whose target (item, category, duration) is that of a row drawn with
        `random.randint(0, n - 1)`, redrawn while the drawn item is in `item_list[i // 5 : i // 5 + 5]` (sic, IT:949);
        negatives carry labels 0 / 0 / 0 and the positive's history.  With ngs = 4 a listwise group of 5 rows is one positive
        and its four negatives.  (The block forgets `item_loop_times_history`; it is replicated like the other histories.)"""
        n = int(res["items"].shape[0])
        if n < self.BEGIN_HISTORY_LEN_MAX:                                   # IT:802-804 returns None
            return {}
        items, cates, durs = res["items"], res["cates"], res["durations"]
        item_list = items.tolist()
        src = np.empty(n * (ngs + 1), np.int64)                              # row whose target each output row takes
        distinct = set(item_list)
        for i in range(n):
            src[i * (ngs + 1)] = i
            group = item_list[i // 5: i // 5 + 5]
            if distinct <= set(group):
                return {}            # (a tail batch of one group) no admissible negative exists: the block would spin forever;
                                     # the batch is dropped like the too-short one above - the loops skip empty feeds
            count = 0
            while count < ngs:
                rv = random.randint(0, n - 1)
                if item_list[rv] in group:
                    continue
                count += 1
                src[i * (ngs + 1) + count] = rv
        rep = lambda a: np.repeat(a, ngs + 1, axis=0)
        is_pos = (np.arange(n * (ngs + 1)) % (ngs + 1) == 0)
        lab = lambda a: np.where(is_pos[:, None], rep(a), 0).astype(np.float32)
        out = {k: rep(v) for k, v in res.items()}                            # histories, masks, users: the positive's
        out["labels_satisfied"], out["labels_play"], out["plays"] = lab(res["labels_satisfied"]), lab(res["labels_play"]), lab(res["plays"])
        out["items"], out["cates"], out["durations"] = items[src], cates[src], durs[src]
        return out

    # ------------------------------------------------------------------ native batcher (csrc/batcher.cu)
    def _native_vocab(self, lib_mod):
        """The three vocabularies as (PamrecVocab, keep-alive arrays), or None when one of them is not a plain
        {str: int32} dict (then `dict.get` semantics cannot be reproduced from key bytes and Python parses)."""
        if "_native_vocab_cache" in self.__dict__:
            return self._native_vocab_cache
        out = []
        for d in (self.userdict, self.itemdict, self.catedict):
            ok = type(d) is dict and all(type(k) is str for k in d) and all(type(v) is int and -2 ** 31 <= v < 2 ** 31 for v in d.values())
            if ok:
                try:
                    keys = [k.encode("utf-8") for k in d]
                except UnicodeEncodeError:
                    ok = False
            if not ok:
                out = None
                break
            blob = np.frombuffer(b"".join(keys) or b"\0", np.uint8)
            offs = np.concatenate([[0], np.cumsum([len(k) for k in keys])]).astype(np.int64)
            vals = np.fromiter(d.values(), np.int32, len(d))
            out.append((lib_mod.PamrecVocab(n=len(d), bytes=blob.ctypes.data, offsets=offs.ctypes.data, values=vals.ctypes.data),
                        (blob, offs, vals)))
        self._native_vocab_cache = out
        return out

    def _tokenize_native(self, infile, train):
        """Flat columns of the file from the native tokenizer (csrc/tokenizer.cu), or None when the file (or the configuration)
        is outside what it converts bit-identically to `parser_one_line` - then the Python parser runs."""
        if os.environ.get("PAMREC_PY_TOKENIZER", "0") == "1" or self.noise_only_predict != 0 or self.col_spliter != "\t":
            return None
        from . import _lib
        lib = _lib.load()
        voc = self._native_vocab(_lib)
        if voc is None:
            return None
        handle, n_lines, n_tok = C.c_void_p(), C.c_int64(), C.c_int64()
        rc = lib.pamrec_tokenize_file(os.fsencode(infile), int(train), C.byref(voc[0][0]), C.byref(voc[1][0]), C.byref(voc[2][0]),
                                      int(os.environ.get("PAMREC_TOKENIZER_THREADS", "0")), C.byref(handle), C.byref(n_lines), C.byref(n_tok))
        if rc == -2:
            raise FileNotFoundError(infile)      # what open() raises in parse_file
        if rc != 0:
            return None
        try:
            n, m = n_lines.value, n_tok.value
            col = {"offsets": np.empty(n + 1, np.int64), "items": np.empty(m, np.int32), "cates": np.empty(m, np.int32),
                   "durs": np.empty(m, np.float64), "sats": np.empty(m, np.float64), "plays": np.empty(m, np.float64),
                   "user_ids": np.empty(n, np.int32)}
            if not train:
                col.update(label_sat=np.empty(n, np.float64), label_play=np.empty(n, np.float64), tgt_item=np.empty(n, np.int32),
                           tgt_cate=np.empty(n, np.int32), tgt_dur=np.empty(n, np.float64))
            desc = _lib.PamrecLines(n_lines=n, **{k: v.ctypes.data for k, v in col.items()})
            if lib.pamrec_tokens_read(handle, C.byref(desc)) != 0:
                raise RuntimeError("pamrec_tokens_read failed")
        finally:
            lib.pamrec_tokens_free(handle)
        return col

    def _flatten(self, lines, train):
        """The same columns from lines parsed in Python; None for ragged history columns (the reference zips them)."""
        h = 1 if train else 6                                        # first history column inside a parsed line
        rows = [ln for ln in lines if ln]
        lens = [len(ln[h]) for ln in rows]
        if any(not (len(ln[h + 1]) == len(ln[h + 2]) == len(ln[h + 3]) == len(ln[h + 4]) == n) for ln, n in zip(rows, lens)):
            return None
        cat = lambda j, dt: (np.concatenate([np.asarray(ln[j], dtype=dt) for ln in rows]) if rows else np.zeros(0, dt))
        col = {"offsets": np.concatenate([[0], np.cumsum(lens)]).astype(np.int64), "items": cat(h, np.int32), "cates": cat(h + 1, np.int32),
               "durs": cat(h + 2, np.float64), "sats": cat(h + 3, np.float64), "plays": cat(h + 4, np.float64)}
        if train:
            col["user_ids"] = np.asarray([ln[0] for ln in rows], np.int32)
        else:
            col["user_ids"] = np.asarray([ln[2] for ln in rows], np.int32)
            col["label_sat"] = np.asarray([ln[0] for ln in rows], np.float64)
            col["label_play"] = np.asarray([ln[1] for ln in rows], np.float64)
            col["tgt_item"] = np.asarray([ln[3] for ln in rows], np.int32)
            col["tgt_cate"] = np.asarray([ln[4] for ln in rows], np.int32)
            col["tgt_dur"] = np.asarray([ln[5] for ln in rows], np.float64)
        return col

    def _native(self, infile, train):
        """Flat columns + a pamrec_batcher handle for this file, or None when the pure-Python path must be used."""
        if os.environ.get("PAMREC_PY_ITERATOR", "0") == "1":
            return None
        if self.noise_train_hist != 0 or self.noise_train_listwise != 0 or self.batch_size % 5:
            return None
        cache = self.__dict__.setdefault("_native_cache", {})
        key = (infile, train)
        if key in cache:
            return cache[key]
        from . import _lib
        lib = _lib.load()
        col = self._tokenize_native(infile, train)
        if col is None:
            col = self._flatten(self._lines(infile), train)
        if col is None:
            cache[key] = None
            return None
        n = len(col["user_ids"])
        desc = _lib.PamrecLines(n_lines=n, **{k: v.ctypes.data for k, v in col.items()})
        borders = np.asarray(_borders(self.dataset, self.bucket_num), np.float64)
        handle = C.c_void_p()
        if lib.pamrec_batcher_create(C.byref(desc), borders.ctypes.data, len(borders), self.max_seq_length, C.byref(handle)) != 0:
            raise RuntimeError("pamrec_batcher_create failed")
        nat = dict(lib=lib, handle=handle, col=col, borders=borders, desc=desc, n=n)
        if train:
            off = col["offsets"]
            nonempty = off[1:] > off[:-1]
            nat["sat_num"] = np.zeros(n)
            if nonempty.any():                                       # sum(sats) per line, in file order like the builtin
                nat["sat_num"][nonempty] = np.add.reduceat(col["sats"], off[:-1][nonempty])
        cache[key] = nat
        return nat

    _FEED_DTYPES = (np.float32, np.float32, np.float32, np.float32, np.int32, np.int32, np.float32, np.int32, np.int32,
                    np.float32, np.float32, np.float32, np.float32, np.float32, np.int32, np.int32, np.float32, np.float32, np.float32)

    def _native_batches(self, nat, train, shard=None):
        """shard = (world, rank): every rank draws the same global batches but materialises only the rows it trains on / scores
        (``LocalFeed``; groups of 5 stay whole in training batches, pamrec_b200/dist.py split_feed is the same selection)."""
        T, bs = self.max_seq_length, self.batch_size
        cap = bs
        if shard:
            world, rank = shard
            cap = max(-(-(bs // 5) // world) * 5 if train else -(-bs // world), 1)
        while True:
            arrs = [np.empty((cap, T) if i >= 7 else ((cap, 1) if i < 3 else (cap,)), dt) for i, dt in enumerate(self._FEED_DTYPES)]
            ptrs = (C.c_void_p * 19)(*[a.ctypes.data for a in arrs])
            if shard:
                g_lab, g_usr, g_rows = np.empty(bs, np.float32), np.empty(bs, np.float32), C.c_int(0)
                n = nat["lib"].pamrec_batcher_next_shard(nat["handle"], bs, world, rank, ptrs, g_lab.ctypes.data, g_usr.ctypes.data,
                                                         C.byref(g_rows))
                total = g_rows.value
            else:
                total = n = nat["lib"].pamrec_batcher_next(nat["handle"], bs, ptrs)
            if n < 0:
                raise RuntimeError(f"pamrec_batcher_next failed ({n})")
            if total == 0:
                return
            feed = {k: (a if n == cap else a[:n]) for k, a in zip(FEED_KEYS, arrs)}
            if shard:
                feed = LocalFeed(feed)
                feed.global_rows, feed.world, feed.rank = total, world, rank
                feed.global_labels_satisfied, feed.global_users = g_lab[:total].reshape(-1, 1), g_usr[:total]
            yield feed

    def _train_batches_native(self, nat, shard=None):
        G = self.BEGIN_HISTORY_LEN_MAX
        order, begin = [], []
        for idx, sn in enumerate(nat["sat_num"]):                    # file order: the RNG call sequence of IT:538-545
            if sn < 2:
                continue
            begin.append(1 if sn <= G else random.randint(1, G))
            order.append(idx)
        pairs = list(zip(order, begin))
        random.shuffle(pairs)                                        # IT:622 (a shuffle permutes by position only)
        order = np.asarray([p[0] for p in pairs], np.int64)
        begin = np.asarray([p[1] for p in pairs], np.int32)
        if nat["lib"].pamrec_batcher_begin_train(nat["handle"], order.ctypes.data, begin.ctypes.data, len(order)) != 0:
            raise RuntimeError("pamrec_batcher_begin_train failed")
        yield from self._native_batches(nat, True, shard)

    def _eval_batches_native(self, nat, min_seq_length, shard=None):
        if nat["lib"].pamrec_batcher_begin_eval(nat["handle"], int(min_seq_length)) != 0:
            raise RuntimeError("pamrec_batcher_begin_eval failed")
        yield from self._native_batches(nat, False, shard)

    def _new_acc(self):
        return {"sat": [], "lplay": [], "plays": [], "users": [], "items": [], "cates": [], "durs": [], "hist": []}

    def _eval_batches(self, lines, min_seq_length):
        acc = self._new_acc()
        for line in lines:
            if not line:
                continue
            (label_satisfied, label_play, user_id, item_id, item_cate, duration, items, cates, durs, sats, plays) = line
            if len(items) < min_seq_length:
                continue
            acc["sat"].append(label_satisfied)
            acc["lplay"].append(1.0 if label_play >= 10 else 0.0)       # IT:410 (10 s at eval, 8 s at train)
            acc["plays"].append(label_play)                             # IT:411 seconds, not a bucket
            acc["users"].append(user_id)
            acc["items"].append(item_id)
            acc["cates"].append(item_cate)
            acc["durs"].append(duration)
            n = min(len(plays), len(durs))
            loops = lisan_array(_ratio64(plays[:n], durs[:n]), self.dataset, self.bucket_num)   # IT:421
            acc["hist"].append((items, cates, durs, sats, plays, loops, 1))
            if len(acc["sat"]) == self.batch_size:
                yield self._convert_data(acc)
                acc = self._new_acc()
        if acc["sat"]:
            yield self._convert_data(acc)

    def _push(self, st, item, cate, dur, sat, play):
        """add_a_item_to_hist (IT:479-522).  st = [items, cates, durs, sats, plays, not_satisfied_index]."""
        if play < self.VALID_THRESHOLD and sat != 1:
            return
        items, cates, durs, sats, plays, nsi = st
        items.append(item); cates.append(cate); durs.append(dur); sats.append(sat)
        plays.append(play if self.noise_train_hist == 0 else max(play + np.random.normal(0, self.noise_train_hist), 0))
        if sat == 0:
            nsi.append(len(items) - 1)
        if len(items) > self.MAX_SEQUENCE:
            if not nsi:
                for col in (items, cates, durs, sats, plays):
                    del col[:-self.MAX_SEQUENCE]
            else:
                k = len(items) - self.MAX_SEQUENCE
                for j, idx in enumerate(nsi[:k]):      # evict the oldest unsatisfied first
                    for col in (items, cates, durs, sats, plays):
                        col.pop(idx - j)
                st[5] = [i - k for i in nsi[k:]]

    def _train_batches(self, lines):
        G = self.BEGIN_HISTORY_LEN_MAX
        data_source = []
        for line in lines:
            if not line:
                continue
            user_id, items, cates, durs, sats, plays = line
            satisfied_num = sum(sats)
            if satisfied_num < 2:
                continue
            begin_loc = 1 if satisfied_num <= G else random.randint(1, G)       # IT:542-545
            st = [[], [], [], [], [], []]
            i = 0
            while sats[i] != 1:                                                 # IT:556-570
                self._push(st, items[i], cates[i], durs[i], sats[i], plays[i])
                i += 1
            for _ in range(begin_loc):                                          # IT:573-588
                self._push(st, items[i], cates[i], durs[i], sats[i], plays[i])
                i += 1
            data_source.append([st, user_id, i, line])
        random.shuffle(data_source)                                             # IT:622
        acc = self._new_acc()
        alive = list(range(len(data_source)))
        while alive:
            nxt = []
            for ind in alive:
                st, user_id, i, line = data_source[ind]
                _, items, cates, durs, sats, plays = line
                future = len(items) - i
                if future < G:
                    continue
                fplays = plays[i:i + G]
                fdurs = durs[i:i + G]
                acc["sat"].extend(sats[i:i + G])
                acc["lplay"].extend(1.0 if x >= self.VALID_THRESHOLD else 0.0 for x in fplays)     # IT:646
                if self.noise_train_listwise == 0:
                    ratio = _ratio64(fplays, fdurs)
                else:                                                                               # IT:656
                    ratio = _ratio64([max(x + np.random.normal(0, self.noise_train_listwise), 0) for x in fplays], fdurs)
                acc["plays"].extend(lisan_array(ratio, self.dataset, self.bucket_num).tolist())
                acc["users"].extend([user_id] * G)
                acc["items"].extend(items[i:i + G])
                acc["cates"].extend(cates[i:i + G])
                acc["durs"].extend(fdurs)
                h_items, h_cates, h_durs, h_sats, h_plays, _ = st
                loops = lisan_array(_ratio64(h_plays, h_durs), self.dataset, self.bucket_num)       # IT:682
                acc["hist"].append((list(h_items), list(h_cates), list(h_durs), list(h_sats), list(h_plays), loops, G))
                if len(acc["sat"]) == self.batch_size:                                              # IT:684-685
                    yield self._convert_data(acc)
                    acc = self._new_acc()
                if future > G:                                                                      # IT:719-741
                    for k in range(i, i + G):
                        self._push(st, items[k], cates[k], durs[k], sats[k], plays[k])
                    data_source[ind][2] = i + G
                    nxt.append(ind)
            alive = nxt
        if acc["sat"]:                                                                              # IT:745-763
            yield self._convert_data(acc)

    # ------------------------------------------------------------------ arrays (IT:1009-1141, no-negatives branch)
    def _convert_data(self, acc):
        T = self.max_seq_length
        n = len(acc["sat"])
        item_h = np.zeros((n, T), np.int32)
        cate_h = np.zeros((n, T), np.int32)
        dur_h = np.zeros((n, T), np.float32)
        sat_h = np.zeros((n, T), np.float32)
        play_h = np.zeros((n, T), np.float32)
        loop_h = np.zeros((n, T), np.float32)
        mask = np.zeros((n, T), np.float32)
        r = 0
        for items, cates, durs, sats, plays, loops, rep in acc["hist"]:
            L = min(len(items), T)
            if L:
                rows = slice(r, r + rep)
                item_h[rows, :L] = items[-L:]
                cate_h[rows, :L] = cates[-L:]
                dur_h[rows, :L] = durs[-L:]
                sat_h[rows, :L] = sats[-L:]
                play_h[rows, :L] = plays[-L:]
                loop_h[rows, :L] = loops[-L:]
                mask[rows, :L] = 1.0
            r += rep
        # satisfied-only compaction (IT:1069-1103); the bucket here comes from the float32 arrays
        is_sat = (sat_h == 1.0) & (mask == 1.0)
        order = np.argsort(~is_sat, axis=1, kind="stable")
        cnt = is_sat.sum(1)
        keep = np.arange(T)[None, :] < cnt[:, None]
        take = lambda a: np.where(keep, np.take_along_axis(a, order, 1), 0)
        with np.errstate(divide="ignore", invalid="ignore"):
            sat_loops = lisan_array(play_h / dur_h, self.dataset, self.bucket_num).astype(np.float32)
        res = {
            "labels_satisfied": np.asarray(acc["sat"], dtype=np.float32).reshape(-1, 1),
            "labels_play": np.asarray(acc["lplay"], dtype=np.float32).reshape(-1, 1),
            "plays": np.asarray(acc["plays"], dtype=np.float32).reshape(-1, 1),
            "users": np.asarray(acc["users"], dtype=np.float32),          # IT:1115 builds users as float32
            "items": np.asarray(acc["items"], dtype=np.int32),
            "cates": np.asarray(acc["cates"], dtype=np.int32),
            "durations": np.asarray(acc["durs"], dtype=np.float32),
            "item_history": item_h,
            "item_cate_history": cate_h,
            "item_duration_history": dur_h,
            "mask": mask,
            "item_satisfied_value_history": sat_h,
            "item_play_value_history": play_h,
            "item_loop_times_history": loop_h,
            "satisfied_item_history": take(item_h).astype(np.int32),
            "satisfied_cate_history": take(cate_h).astype(np.int32),
            "satisfied_duration_history": take(dur_h).astype(np.float32),
            "satisfied_play_history": take(sat_loops).astype(np.float32),
            "satisfied_mask": keep.astype(np.float32),
        }
        return res

    def item_categories(self, files):
        """Item -> category table [n_items] int32 from the target and history columns of ``files`` (the mode of each file follows
        its basename, as in load_data_from_file): the first occurrence in file order wins (in an evaluation line the target comes
        before the history); items that never appear get -1, and so does item 0 (padding / unknown)."""
        table = np.full(len(self.itemdict), -1, np.int32)
        for infile in files:
            train = os.path.basename(infile) == "train_data"
            col = self._tokenize_native(infile, train)
            if col is None:
                self.train = train
                col = self._flatten(self._lines(infile), train)
            if col is not None:
                items, cates = col["items"], col["cates"]
                if not train:
                    starts = col["offsets"][:-1]
                    items, cates = np.insert(items, starts, col["tgt_item"]), np.insert(cates, starts, col["tgt_cate"])
            else:                                                    # ragged history columns: pairs as far as both go
                h = 1 if train else 6
                items, cates = [], []
                for ln in self._lines(infile):
                    if not ln:
                        continue
                    pairs = ([(ln[3], ln[4])] if not train else []) + list(zip(ln[h], ln[h + 1]))
                    items.extend(p[0] for p in pairs)
                    cates.extend(p[1] for p in pairs)
            items = np.asarray(items, np.int64)
            ok = (items >= 0) & (items < table.size)
            items, cates = items[ok], np.asarray(cates, np.int64)[ok]
            uniq, first = np.unique(items, return_index=True)
            new = table[uniq] < 0
            table[uniq[new]] = cates[first[new]]
        if table.size:
            table[0] = -1
        return table

    def gen_feed_dict(self, data_dict):
        """IT:1143-1181: identity here — the feed mapping is keyed by placeholder name."""
        return {k: data_dict[k] for k in FEED_KEYS}
