"""foodrec_b200 -- B200-native hot path of Market2Dish's Code/Recommender.

Public surface mirrors the reference: ``Model`` (Model_Recommender.py:5),
``evaluate_model`` (evaluate.py:13) and its full-ranking counterpart
``evaluate_full_catalog``, its row-sharded form ``evaluate_sharded``, a ``Session``/``Saver`` shim for
Train_recommender.py, and the explicit ``Engine`` underneath.  Importing the package
needs neither a GPU nor the built library; using it needs both (no fallback).
"""
from .data import Dataset, InstanceStream, build_instances
from .engine import Engine, Hyper, history_csr
from .evaluate import evaluate_full_catalog, evaluate_model, evaluate_sharded
from .model import ConfigProto, Model, Saver, Session, global_variables_initializer, latest_checkpoint

__all__ = ["Engine", "Hyper", "Model", "Session", "Saver", "ConfigProto", "evaluate_model", "evaluate_full_catalog",
           "evaluate_sharded", "Dataset", "InstanceStream", "history_csr",
           "build_instances",
           "global_variables_initializer", "latest_checkpoint"]
