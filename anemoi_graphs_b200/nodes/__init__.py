from .builders.from_file import LimitedAreaNPZFileNodes
from .builders.from_file import NPZFileNodes
from .builders.from_file import TextNodes
from .builders.from_file import ZarrDatasetNodes
from .builders.from_healpix import HEALPixNodes
from .builders.from_healpix import LimitedAreaHEALPixNodes
from .builders.from_reduced_gaussian import ReducedGaussianGridNodes
from .builders.from_refined_icosahedron import HexNodes
from .builders.from_refined_icosahedron import LimitedAreaHexNodes
from .builders.from_refined_icosahedron import LimitedAreaTriNodes
from .builders.from_refined_icosahedron import StretchedTriNodes
from .builders.from_refined_icosahedron import TriNodes
from .builders.from_vectors import LatLonNodes

__all__ = [
    "ZarrDatasetNodes",
    "NPZFileNodes",
    "TriNodes",
    "HexNodes",
    "HEALPixNodes",
    "LatLonNodes",
    "LimitedAreaHEALPixNodes",
    "ReducedGaussianGridNodes",
    "LimitedAreaNPZFileNodes",
    "LimitedAreaTriNodes",
    "LimitedAreaHexNodes",
    "StretchedTriNodes",
    "TextNodes",
]
