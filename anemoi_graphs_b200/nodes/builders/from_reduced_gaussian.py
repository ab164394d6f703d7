"""Nodes of a named reduced Gaussian grid (``ReducedGaussianGridNodes`` of newer anemoi-graphs releases).

Upstream reads the coordinates of the named grid from a downloaded ``grid-<name>.npz``.  An octahedral grid O<N> is
defined by its construction - the 2N Gaussian latitudes, and 4i + 16 equally spaced longitudes from 0 degrees on row i
counted from the nearer pole - so here two kernels compute it (``ops.octahedral_nodes``), bit for bit the values of
``grids.latlon_deg_to_x(*grids.octahedral_grid(N))``.  Classic N grids take their per-row counts from ECMWF's ``pl``
tables, which this package does not have: they raise NotImplementedError."""

from __future__ import annotations

import logging
import re

import torch

from ... import device as _device
from ... import ops
from .base import BaseNodeBuilder

LOGGER = logging.getLogger(__name__)


def octahedral_number(grid) -> int:
    """N of an octahedral grid name ``"o<N>"`` / ``"O<N>"``, N >= 1.  AssertionError for anything that is not a reduced
    Gaussian grid name, NotImplementedError for a classic ``"n<N>"`` / ``"N<N>"`` grid."""
    assert isinstance(grid, str), f"Grid {grid!r} must be a string, such as 'o96'."
    match = re.fullmatch(r"([nNoO])([0-9]+)", grid)
    assert match is not None and int(match.group(2)) >= 1, f"Grid {grid!r} is not a valid reduced Gaussian grid."
    if match.group(1) in "nN":
        raise NotImplementedError(
            f"Grid {grid!r}: classic reduced Gaussian grids need ECMWF's per-row point counts, which are not built; "
            "octahedral grids ('o<N>') are."
        )
    return int(match.group(2))


class ReducedGaussianGridNodes(BaseNodeBuilder):
    """Nodes from a reduced Gaussian grid.

    Attributes
    ----------
    grid : str
        The grid name: ``"o<N>"`` or ``"O<N>"``, the octahedral grid with N latitudes between a pole and the equator.
    """

    def __init__(self, grid: str, name: str) -> None:
        self.n = octahedral_number(grid)
        self.grid = grid
        super().__init__(name)

    def get_coordinates(self) -> torch.Tensor:
        """float32 (4N(N + 9), 2) coordinates of the nodes, in radians."""
        LOGGER.info(f"Creating reduced Gaussian grid nodes of grid O{self.n}.")
        self._x_device = ops.octahedral_nodes(self.n)
        return self._x_device if _device.is_resident() else _device.to_host(self._x_device)

    def register_nodes(self, graph):
        graph = super().register_nodes(graph)
        _device.seed_node_state(graph[self.name], self._x_device)
        _device.maybe_flush()
        return graph
