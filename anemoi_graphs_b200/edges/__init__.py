from .builder import CutOffEdges
from .builder import KNNEdges
from .builder import MultiScaleEdges
from .builder import ReversedCutOffEdges
from .builder import ReversedKNNEdges

__all__ = ["KNNEdges", "CutOffEdges", "MultiScaleEdges", "ReversedKNNEdges", "ReversedCutOffEdges"]
