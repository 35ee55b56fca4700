"""Drop-in for the reference graph object and its session protocol.

``Model(args, Personal_Memory, Recipe_Embedding, Category_Embedding, General_Memory)``
keeps the constructor, the feed handles (``user_input, item_input, labels, write_sign,
categories, user_one_hot_label, dropout_keep_prob, is_training_flag`` --
Model_Recommender.py:26-35) and the fetch handles (``logits, loss_value, personal,
general, train_op, learning_rate, epoch_step, epoch_increment`` -- :14-16,38-41) of
``/root/reference/Code/Recommender/Model_Recommender.py``.  ``Session.run(fetches,
feed_dict)`` maps the three fetch patterns of ``Train_recommender.py:182-186,195-199``
and ``evaluate.py:58`` onto the CUDA engine; fetching ``personal`` is what makes a
step a personal-memory write step, exactly as in the reference graph.
"""
from __future__ import annotations

import glob
import os

import numpy as np

from . import _lib as L
from .engine import Engine, Hyper


class Handle:
    """Opaque token standing in for a tf.placeholder / fetchable tensor."""
    __slots__ = ("name", "kind", "model")

    def __init__(self, name, kind, model=None):
        self.name, self.kind, self.model = name, kind, model

    def __repr__(self):
        return f"<foodrec_b200 {self.kind} '{self.name}'>"

    def __hash__(self):
        return id(self)

    def __eq__(self, other):
        return self is other


class Model:
    def __init__(self, args, Personal_Memory, Recipe_Embedding, Category_Embedding, General_Memory,
                 device="cuda:0", max_batch=None, adam_mode="lazy"):
        self.learner = args.learner
        self.num_categories = args.num_categories
        self.num_users = args.num_users
        self.num_labels = args.num_labels
        self.embed_size = args.embed_size
        self.decay_steps = getattr(args, "decay_steps", 1000)
        self.decay_rate = getattr(args, "decay_rate", 1.0)
        self.beta_1, self.beta_2, self.alpha = args.beta_1, args.beta_2, args.alpha
        if self.num_categories != 4:
            raise ValueError("num_categories is hard-wired to 4 by tf.split(..., [1, 4]) "
                             "(Model_Recommender.py:59-60)")
        P = np.asarray(Personal_Memory); R = np.asarray(Recipe_Embedding)
        Cat = np.asarray(Category_Embedding); G = np.asarray(General_Memory)
        for name, t in (("Personal_Memory", P), ("Recipe_Embedding", R),
                        ("Category_Embedding", Cat), ("General_Memory", G)):
            if t.dtype != np.float32:
                raise TypeError(f"{name} must be float32 (the reference multiplies it with float32 "
                                f"placeholders, Model_Recommender.py:32,67); got {t.dtype}")
        if P.shape != (args.num_users, 5, args.embed_size):
            raise ValueError(f"Personal_Memory must be [num_users,5,embed_size], got {P.shape}")
        if G.shape != (args.num_labels, 5, args.embed_size):
            raise ValueError(f"General_Memory must be [num_labels,5,embed_size], got {G.shape}")
        ph = lambda n: Handle(n, "placeholder", self)
        self.user_input, self.item_input, self.labels = ph("user_input"), ph("item_input"), ph("labels")
        self.write_sign, self.categories = ph("write_sign"), ph("categories")
        self.user_one_hot_label = ph("user_labels")
        self.dropout_keep_prob, self.is_training_flag = ph("dropout_keep_prob"), ph("is_training_flag")
        # BPR extension feeds (not in the reference)
        self.neg_item_input, self.neg_categories = ph("neg_item_input"), ph("neg_categories")
        ft = lambda n: Handle(n, "fetch", self)
        self.logits, self.loss_value = ft("logits"), ft("loss_value")
        self.personal, self.general, self.train_op = ft("personal"), ft("general"), ft("train_op")
        self.learning_rate, self.epoch_step, self.epoch_increment = ft("learning_rate"), ft("Epoch_Step"), ft("epoch_increment")
        self.global_step = ft("Global_Step")
        self._epoch = 0
        if max_batch is None:
            max_batch = max(int(getattr(args, "batch_size", 128)), 128)
        self.engine = Engine(Hyper.from_args(args), P, R, Cat, G, device=device, max_rows=2 * max_batch,
                             max_label_entries=2 * max_batch * args.num_labels, adam_mode=adam_mode)
        global _LAST_MODEL
        _LAST_MODEL = self

    # explicit API (what Session.run dispatches to)
    def train_step(self, feed, write_personal=False):
        e = self.engine
        out = e.train_step(feed[self.user_input], feed[self.item_input], labels=feed.get(self.labels),
                           categories=feed[self.categories], write_sign=feed.get(self.write_sign),
                           user_one_hot_label=feed[self.user_one_hot_label],
                           neg_items=feed.get(self.neg_item_input), neg_categories=feed.get(self.neg_categories),
                           write_personal=write_personal)
        return out

    def score(self, feed):
        return self.engine.score(feed[self.user_input], feed[self.item_input], feed[self.categories])

    def catalog_topk(self, user_ids, K, dish_to_category=None, exclude=None):
        """The K best recipes of the WHOLE catalog for each user, by (``model.logits`` desc, id asc) --
        ``evaluate.py:55-63`` with every recipe as a candidate.  ``dish_to_category`` is the reference's
        json map (``Train_recommender.py:132``: item -> [[m0],[m1],[m2],[m3]]); it is only needed on the
        first call or when it changed.  ``exclude``: a dict keyed like ``Dataset.trainMatrix``
        (``str(user)`` -> recipe ids) of recipes a user must not get back, e.g. what they trained on.
        Returns (ids int32 [n,K], scores float64 [n,K]) as numpy; ids of recipes beyond the catalog are -1."""
        e = self.engine
        if dish_to_category is not None:
            ic = np.zeros((e.I, 4), np.float32)
            for it, m in dish_to_category.items():
                if 0 <= int(it) < e.I:
                    ic[int(it)] = np.asarray(m, np.float32).reshape(4)
            e.set_item_cats(ic)
        # (the engine rebuilds its recipe index by itself when a training step has run since)
        users = np.asarray([int(u) for u in user_ids], np.int32)
        ex = None if exclude is None else [[int(i) for i in exclude.get(str(int(u)), ())] for u in users]
        ids, sc = e.catalog_topk(users=users, K=int(K), exclude=ex)
        return ids.cpu().numpy(), sc.cpu().numpy()


class _Initializer:
    pass


def global_variables_initializer():
    return _Initializer()


class ConfigProto:
    def __init__(self, **kw):
        class _GPU:
            allow_growth = False
        self.gpu_options = _GPU()


class Session:
    """``tf.Session`` stand-in: synchronous ``run(fetches, feed_dict)``."""

    def __init__(self, config=None):
        self._model = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False

    def run(self, fetches, feed_dict=None):
        single = not isinstance(fetches, (list, tuple))
        fl = [fetches] if single else list(fetches)
        if len(fl) == 1 and isinstance(fl[0], _Initializer):
            return None
        model = self._find_model(fl, feed_dict)
        self._model = model or self._model
        model = self._model
        if model is None:
            raise RuntimeError("Session.run: cannot tell which Model these handles belong to")
        res = {}
        names = {f.name for f in fl if isinstance(f, Handle)}
        if "train_op" in names:
            model.train_step(feed_dict, write_personal="personal" in names)
            v = model.engine.read_scalars()
            res.update(loss_value=np.float32(v[L.FR_OUT_LOSS]), learning_rate=np.float32(v[L.FR_OUT_LR]),
                       general=np.float32(v[L.FR_OUT_GENERAL]), personal=np.float32(v[L.FR_OUT_PERSONAL]),
                       train_op=None)
        elif names & {"loss_value", "personal", "general"}:
            raise NotImplementedError("fetching loss/personal/general without train_op is not a pattern the "
                                      "reference uses (Train_recommender.py:182-199)")
        if "logits" in names:
            res["logits"] = model.score(feed_dict).cpu().numpy()
        if "learning_rate" in names and "learning_rate" not in res:
            res["learning_rate"] = np.float32(model.engine.h.lr)
        if "Epoch_Step" in names:
            res["Epoch_Step"] = model._epoch
        if "Global_Step" in names:
            res["Global_Step"] = 0      # never incremented: apply_gradients gets no global_step (:240)
        if "epoch_increment" in names:
            model._epoch += 1
            res["epoch_increment"] = model._epoch
        out = [res[f.name] for f in fl]
        return out[0] if single else out

    @staticmethod
    def _find_model(fl, feed):
        for f in list(fl) + list(feed or ()):
            if isinstance(f, Handle) and f.model is not None:
                return f.model
        return None


_LAST_MODEL = None


class Saver:
    """``tf.train.Saver`` stand-in: one ``.npz`` per checkpoint holding the tables, the
    optimizer slots, the step and the epoch counter; writes a ``checkpoint`` index file so
    the reference's ``os.path.exists(dir + "checkpoint")`` test works."""

    def save(self, sess, save_path, global_step=None):
        model = sess._model or _LAST_MODEL
        path = save_path if global_step is None else f"{save_path}-{global_step}"
        sd = model.engine.state_dict()
        sd["epoch"] = np.int64(model._epoch)
        np.savez(path + ".npz", **sd)
        d = os.path.dirname(path) or "."
        with open(os.path.join(d, "checkpoint"), "w") as f:
            f.write(f'model_checkpoint_path: "{os.path.basename(path)}"\n')
        return path

    def restore(self, sess, save_path):
        model = sess._model or _LAST_MODEL
        sd = dict(np.load(save_path + ".npz"))
        model._epoch = int(sd.pop("epoch", 0))
        model.engine.load_state_dict(sd)
        sess._model = model


def latest_checkpoint(checkpoint_dir):
    idx = os.path.join(checkpoint_dir, "checkpoint")
    if os.path.exists(idx):
        line = open(idx).read().strip()
        name = line.split('"')[1] if '"' in line else None
        if name and os.path.exists(os.path.join(checkpoint_dir, name + ".npz")):
            return os.path.join(checkpoint_dir, name)
    cands = sorted(glob.glob(os.path.join(checkpoint_dir, "*.npz")), key=os.path.getmtime)
    return cands[-1][:-4] if cands else None
