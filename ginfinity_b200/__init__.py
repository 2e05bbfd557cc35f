"""ginfinity_b200 -- B200-native GINFINITY encoder path.

Exports the names a user of the reference package imports for this path
(src/ginfinity/__init__.py:14-36), so `import ginfinity_b200 as ginfinity` is the
whole migration.  The data plane (records, graph specification, graphs,
shards and their files) is importable anywhere; `Ginfinity`, `DeviceShard`,
`EmbeddingIndex`, `align_pairs` and `align_paths` need the built libgfx.so and a CUDA device and are resolved on
first use -- they fail loudly without them, there is no CPU fallback.
"""
import importlib

from . import graph as _graph
from . import records as _records
from . import weights as _weights

__version__ = "0.1.0"

# module -> names re-exported from it (eagerly: plain NumPy host code)
_EAGER = {
    _records: ("InputValidationError", "RNA", "read_rna_table"),
    _graph: ("GRAPH_SHARD_FORMAT", "GRAPH_SHARD_FORMAT_VERSION", "NODE_ROLE_CONTEXT", "NODE_ROLE_CORE",
             "Graph", "GraphBuilder", "GraphCompatibilityError", "GraphShard", "GraphSpec",
             "GraphValidationError", "graph_metadata_path", "load_graph_shard", "partition_records",
             "save_graph_shard"),
    _weights: ("EncoderConfig", "ModelIntegrityError"),
}
# name -> submodule that is imported only when the name is first touched (needs the GPU library)
_LAZY = {"Ginfinity": "encoder", "DeviceShard": "encoder", "default_alignment_parameters": "encoder",
         "EmbeddingIndex": "search", "align_pairs": "align", "Alignments": "align",
         "align_paths": "align", "AlignmentPaths": "align"}

for _module, _names in _EAGER.items():
    for _name in _names:
        globals()[_name] = getattr(_module, _name)


def __getattr__(name):
    target = _LAZY.get(name)
    if target is None:
        raise AttributeError(f"module {__name__!r} has no attribute {name!r}")
    return getattr(importlib.import_module(f"{__name__}.{target}"), name)


__all__ = sorted([n for names in _EAGER.values() for n in names] + list(_LAZY)) + ["__version__"]
