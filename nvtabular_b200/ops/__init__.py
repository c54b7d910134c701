"""Hot-path operators with the reference's names and kwargs
(reference nvtabular/ops/__init__.py:21-54; scope per SURVEY.md §8)."""
from .base import Operator, StatOperator  # noqa: F401
from .categorify import Categorify  # noqa: F401
from .clip_log import Clip, LogOp  # noqa: F401
from .fill import FillMissing  # noqa: F401
from .groupby import Groupby  # noqa: F401
from .hash_bucket import HashBucket, emb_sz_rule  # noqa: F401
from .join_groupby import JoinGroupby  # noqa: F401
from .list_slice import ListSlice  # noqa: F401
from .normalize import Normalize, NormalizeMinMax  # noqa: F401
from .target_encoding import TargetEncoding  # noqa: F401


def get_embedding_sizes(source, output_dtypes=None):
    """reference nvtabular/ops/categorify.py:616-663: {column: (cardinality, dimension)}
    from a fitted Workflow or a graph node."""
    from ..graph import Tags
    from ..workflow import Workflow
    node = source.output_node if isinstance(source, Workflow) else source
    schema = source.output_schema if isinstance(source, Workflow) else node.output_schema
    if schema is None:
        raise ValueError("fit the workflow before asking for embedding sizes")
    output, multihot = {}, set()
    for cs in schema.select_by_tag(Tags.CATEGORICAL):
        sizes = cs.properties.get("embedding_sizes", {})
        if not sizes:
            continue
        if cs.is_list and cs.is_ragged:
            multihot.add(cs.name)
        output[cs.name] = (sizes["cardinality"], sizes["dimension"])
    if not multihot:
        return output
    return ({k: v for k, v in output.items() if k not in multihot},
            {k: v for k, v in output.items() if k in multihot})
