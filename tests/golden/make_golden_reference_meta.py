"""
Generates the facts about the UNMODIFIED reference (imported through oracle/ref_import.py) that the CPU tests compare against:

  reference_managers.json     for each shipped retrieval config (config/retrieval/paper2020/*.yaml): every config value that the
                              drop-in RetrievalModelManager reads (recorded while it is constructed from the reference's own
                              RetrievalConfig), and the reference RetrievalModelManager's state-dict inventory (name, shape,
                              dtype per net), optimizer parameter groups and autocast flags; under "dims_64_96" the inventory of
                              the anet manager built with 64 / 96 input dims (oracle/ref_import.make_reference_manager)
  reference_line_counts.json  the line count of every .py / .yaml file under the directories that source citations name

Run where the reference tree is available:  python tests/golden/make_golden_reference_meta.py
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref_import  # noqa: E402
from tests.test_citations import CITED_DIRS  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
CONFIGS = ("anet_coot.yaml", "yc2_100m_coot.yaml", "yc2_2d3d_coot.yaml")


class Recorder:
    """Wraps a config object and records every value read through it: attributes as keys, items under "__items__"."""

    def __init__(self, obj, store):
        self._obj, self._store = obj, store

    def _wrap(self, value, store, key):
        if value is None or isinstance(value, (bool, int, float, str)):
            store[key] = value
            return value
        return Recorder(value, store.setdefault(key, {}))

    def __getattr__(self, key):
        return self._wrap(getattr(self._obj, key), self._store, key)

    def __getitem__(self, key):
        return self._wrap(self._obj[key], self._store.setdefault("__items__", {}), key)


def inventory(mgr):
    return {net: [[k, list(v.shape), str(v.dtype)] for k, v in sd.items()] for net, sd in mgr.get_model_state().items()}


def managers(ns):
    from coot_videotext_b200.model_retrieval import RetrievalModelManager
    out = {}
    for yaml_name in CONFIGS:
        d = ns.load_yaml_config_file(os.path.join(ref_import.REFERENCE_ROOT, "config/retrieval/paper2020", yaml_name))
        d.update(use_cuda=False)
        cfg = ns.RetrievalConfig(d)
        ref = ns.RetrievalModelManager(cfg)
        reads = {}
        mine = RetrievalModelManager(Recorder(cfg, reads))
        mine.get_all_params()
        autocast = {}
        for mode, switch in (("train", "set_all_models_train"), ("eval", "set_all_models_eval")):
            getattr(ref, switch)()
            getattr(mine, switch)()
            autocast[mode] = ref.is_autocast_enabled()
            mine.is_autocast_enabled()
        groups, names, _ = ref.get_all_params()
        out[yaml_name] = {"config_reads": reads, "nets": list(ref.model_dict), "state": inventory(ref), "autocast": autocast,
                          "param_groups": [[n, g["decay_mult"], g["lr_mult"], list(g["params"].shape)] for n, g in zip(names, groups)]}
    _, mgr = ref_import.make_reference_manager(ns, 64, 96)
    out["dims_64_96"] = {"state": inventory(mgr)}
    return out


def line_counts():
    counts = {}
    for top in CITED_DIRS:
        for root, dirs, files in os.walk(os.path.join(ref_import.REFERENCE_ROOT, top)):
            dirs[:] = sorted(d for d in dirs if d != "__pycache__")
            for f in sorted(files):
                if f.endswith((".py", ".yaml")):
                    full = os.path.join(root, f)
                    counts[os.path.relpath(full, ref_import.REFERENCE_ROOT)] = sum(1 for _ in open(full, encoding="utf8", errors="replace"))
    return counts


def _fmt(obj, depth=0):
    """JSON with one dict key per line and every list of scalars / short lists (one inventory entry) on one line."""
    pad = " " * (depth + 1)
    if isinstance(obj, dict):
        items = [f"{pad}{json.dumps(k)}: {_fmt(obj[k], depth + 1)}" for k in sorted(obj)]
        return "{\n" + ",\n".join(items) + "\n" + pad[:-1] + "}" if items else "{}"
    if isinstance(obj, list) and any(isinstance(x, (dict, list)) and any(isinstance(y, (dict, list)) for y in x) for x in obj):
        return "[\n" + ",\n".join(pad + _fmt(x, depth + 1) for x in obj) + "\n" + pad[:-1] + "]"
    return json.dumps(obj)


def dump(obj, name):
    path = os.path.join(HERE, name)
    with open(path, "w") as f:
        f.write(_fmt(obj) + "\n")
    print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    dump(managers(ref_import.import_reference()), "reference_managers.json")
    dump(line_counts(), "reference_line_counts.json")
