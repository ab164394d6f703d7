from .post_process import RemoveUnconnectedNodes
from .post_process import RestrictEdgeLength
from .post_process import SortEdgeIndexBySourceNodes
from .post_process import SortEdgeIndexByTargetNodes

__all__ = ["RemoveUnconnectedNodes", "RestrictEdgeLength", "SortEdgeIndexBySourceNodes", "SortEdgeIndexByTargetNodes"]
