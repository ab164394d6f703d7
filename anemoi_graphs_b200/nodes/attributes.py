"""Node attributes (/root/reference/src/anemoi/graphs/nodes/attributes.py:34-316).

Same class names, constructor arguments and ``compute(graph, nodes_name)`` contract as the reference.  The expensive
one - ``SphericalAreaWeights``, scipy's ``SphericalVoronoi`` over every node (minutes for the 6.6 M nodes of an O1280
grid) - runs on the GPU (``ops.voronoi_areas``: neighbour search + one thread per Voronoi cell); normalisation follows
``normalise.py:20-55`` in float64 on the device.  The masks are elementwise.  Attributes that read Zarr datasets or
need qhull's randomised joggling are not built (they are not on the edge-construction path and have no
deterministic reference output).
"""

from __future__ import annotations

import logging
from abc import ABC
from abc import abstractmethod
from typing import Type
from typing import Union

import numpy as np
import torch

from .. import device as _device
from .. import ops

LOGGER = logging.getLogger(__name__)

MaskAttributeType = Union[str, Type["BooleanBaseNodeAttribute"]]


def normalise_device(values: torch.Tensor, norm: str | None, who: str) -> torch.Tensor:
    """``NormaliserMixin.normalise`` (normalise.py:20-55) on a float64 CUDA tensor."""
    if norm is None:
        return values
    if norm == "l1":
        return values / values.sum()
    if norm == "l2":
        return values / torch.linalg.norm(values)
    if norm == "unit-max":
        return values / values.max()
    if norm == "unit-range":
        lo, hi = values.min(), values.max()
        return (values - lo) / (hi - lo)
    if norm == "unit-std":
        std = values.std(unbiased=False)
        if float(std.item()) == 0:
            LOGGER.warning(f"Std. dev. of the {who} values is 0. Normalisation is skipped.")
            return values
        return values / std
    raise ValueError(
        f"Attribute normalisation \"{norm}\" is not valid. Options are: 'l1', 'l2', 'unit-max' or 'unit-std'."
    )


_TORCH_DTYPES = {"float32": torch.float32, "float64": torch.float64, "float16": torch.float16, "bool": torch.bool}


class BaseNodeAttribute(ABC):
    """Base class for the weights of the nodes."""

    _agx_device_aware = True

    def __init__(self, norm: str | None = None, dtype: str = "float32") -> None:
        self.norm = norm
        self.dtype = dtype

    @abstractmethod
    def get_raw_values(self, nodes, **kwargs) -> torch.Tensor:
        """float64 (or bool) CUDA tensor of shape (N,) or (N, M)."""

    def post_process(self, values: torch.Tensor) -> torch.Tensor:
        """Post-process the values: (N,) -> (N, 1), normalise, cast (nodes/attributes.py:44-52)."""
        if values.dim() == 1:
            values = values[:, None]
        if values.dtype != torch.bool:
            values = normalise_device(values, self.norm, self.__class__.__name__)
        return values.to(_TORCH_DTYPES[str(self.dtype)])

    def compute(self, graph, nodes_name: str, **kwargs) -> torch.Tensor:
        """Get the nodes attribute: tensor of shape (N, M), on the device ``graph[nodes_name].x`` lives on."""
        nodes = graph[nodes_name]
        out = self.post_process(self.get_raw_values(nodes, **kwargs))
        if nodes["x"].is_cuda and not out.is_cuda:  # masks read from files
            out = out.to(nodes["x"].device)
        res = _device.like_input(out, nodes["x"])
        _device.maybe_flush()
        return res


class UniformWeights(BaseNodeAttribute):
    """Implements a uniform weight for the nodes."""

    def get_raw_values(self, nodes, **kwargs) -> torch.Tensor:
        st = _device.node_state(nodes)
        return torch.ones(int(st.x.shape[0]), dtype=torch.float64, device=st.x.device)


class AreaWeights(BaseNodeAttribute):
    """Implements the area of the nodes as the weights (dispatches on ``flat`` like the reference, :103-129)."""

    def __new__(cls, flat: bool = False, **kwargs):
        logging.warning(
            "Creating %s with flat=%s and kwargs=%s. In a future release, AreaWeights will be deprecated: please use directly PlanarAreaWeights or SphericalAreaWeights.",
            cls.__name__,
            flat,
            kwargs,
        )
        if flat:
            return PlanarAreaWeights(**kwargs)
        return SphericalAreaWeights(**kwargs)


class PlanarAreaWeights(BaseNodeAttribute):
    """2D (lat, lon plane) Voronoi areas - not built: the reference calls qhull with ``QJ`` (randomly joggled input,
    nodes/attributes.py:152), so its own output is not reproducible from run to run."""

    def __init__(self, norm: str | None = None, dtype: str = "float32") -> None:
        super().__init__(norm, dtype)

    def get_raw_values(self, nodes, **kwargs) -> torch.Tensor:
        raise NotImplementedError(
            "PlanarAreaWeights is not built: the reference's values come from qhull's randomised joggling (QJ)."
        )


class SphericalAreaWeights(BaseNodeAttribute):
    """Implements the 3D area of the nodes as the weights (nodes/attributes.py:165-221).

    Attributes
    ----------
    norm : str
        Normalisation of the weights.
    radius : float
        Radius of the sphere.
    centre : np.ndarray
        Centre of the sphere.
    fill_value : float
        Value to fill the empty regions.
    """

    def __init__(
        self,
        norm: str | None = None,
        radius: float = 1.0,
        centre: np.ndarray = np.array([0, 0, 0]),
        fill_value: float = 0.0,
        dtype: str = "float32",
    ) -> None:
        super().__init__(norm, dtype)
        self.radius = radius
        self.centre = centre
        self.fill_value = fill_value

    def get_raw_values(self, nodes, **kwargs) -> torch.Tensor:
        # the generators are latlon_rad_to_cartesian(x) with radius 1 around the origin whatever ``radius`` /
        # ``centre`` say (:200-201): scipy rejects any other sphere
        try:
            radius = float(self.radius)
        except (TypeError, ValueError):
            raise ValueError("`radius` is not a floating point number.") from None  # scipy raises ValueError too
        if abs(radius - 1.0) > 1e-6 or np.abs(np.asarray(self.centre, dtype=np.float64)).max() > 1e-6:
            raise ValueError("Radius inconsistent with generators.")  # scipy.spatial.SphericalVoronoi's message
        st = _device.node_state(nodes)
        result = ops.voronoi_areas(st.x, float(self.radius))
        LOGGER.debug("There are %d of weights.", int(result.shape[0]))
        return result


class IsolatitudeAreaWeights(BaseNodeAttribute):
    """Isolatitude area weights (newer anemoi-graphs releases; not in the pinned reference, upstream parity
    unverified): every node gets the area of its latitude band over the number of nodes in its row - the band bounded
    by the midpoints to the neighbouring rows and by the poles (``ops.isolatitude_areas``, DESIGN.md section 4).
    Suits any node set laid out in latitude rows, limited-area ones included."""

    def get_raw_values(self, nodes, **kwargs) -> torch.Tensor:
        areas, n_rows = ops.isolatitude_areas(_device.node_state(nodes).x)
        LOGGER.debug("%d nodes in %d latitude rows.", int(areas.shape[0]), n_rows)
        return areas


class BooleanBaseNodeAttribute(BaseNodeAttribute, ABC):
    """Base class for boolean node attributes."""

    def __init__(self) -> None:
        super().__init__(norm=None, dtype="bool")


class NonmissingZarrVariable(BooleanBaseNodeAttribute):
    """Mask of valid (not missing) values of a Zarr dataset variable in the first timestep
    (nodes/attributes.py:229-258); reads the dataset through anemoi-datasets."""

    def __init__(self, variable: str) -> None:
        super().__init__()
        self.variable = variable

    def get_raw_values(self, nodes, **kwargs) -> torch.Tensor:
        from .builders.from_file import open_dataset

        assert (
            nodes["node_type"] == "ZarrDatasetNodes"
        ), f"{self.__class__.__name__} can only be used with ZarrDatasetNodes."
        ds = open_dataset(nodes["_dataset"], select=self.variable)[0].squeeze()
        return torch.as_tensor(~np.isnan(np.asarray(ds)))


class CutOutMask(BooleanBaseNodeAttribute):
    """Cut out mask (nodes/attributes.py:261-268): True for the limited-area part of a cutout dataset."""

    def get_raw_values(self, nodes, **kwargs) -> torch.Tensor:
        from .builders.from_file import open_dataset

        assert isinstance(nodes["_dataset"], dict), "The 'dataset' attribute must be a dictionary."
        assert "cutout" in nodes["_dataset"], "The 'dataset' attribute must contain a 'cutout' key."
        num_lam, num_other = open_dataset(nodes["_dataset"]).grids
        return torch.as_tensor(np.array([True] * num_lam + [False] * num_other, dtype=bool))


class BooleanOperation(BooleanBaseNodeAttribute, ABC):
    """Base class for boolean operations."""

    def __init__(self, masks: MaskAttributeType | list[MaskAttributeType]) -> None:
        super().__init__()
        self.masks = masks if isinstance(masks, list) else [masks]

    @staticmethod
    def get_mask_values(mask: MaskAttributeType, nodes, **kwargs) -> torch.Tensor:
        if isinstance(mask, str):
            attributes = nodes[mask]
            if not isinstance(attributes, torch.Tensor):
                attributes = torch.as_tensor(np.asarray(attributes))
            assert (
                attributes.dtype == torch.bool
            ), f"The mask attribute '{mask}' must be a boolean but is {attributes.dtype}."
            return attributes.to(nodes["x"].device)

        return mask.get_raw_values(nodes, **kwargs).to(nodes["x"].device)

    @abstractmethod
    def reduce_op(self, masks: list[torch.Tensor]) -> torch.Tensor: ...

    def get_raw_values(self, nodes, **kwargs) -> torch.Tensor:
        mask_values = [BooleanOperation.get_mask_values(mask, nodes, **kwargs) for mask in self.masks]
        # a stored attribute is (N, 1), a nested mask object's raw values are (N,): mixing them would broadcast to
        # (N, N).  One shape for all; anything that is not one value per node is an error (the reference's
        # ``np.logical_and.reduce`` on such a ragged list raises too).
        n = int(nodes["x"].shape[0])
        flat = []
        for mask, values in zip(self.masks, mask_values):
            if values.dim() == 2 and values.shape[1] == 1:
                values = values.squeeze(-1)
            if values.shape != (n,):
                raise ValueError(f"The mask '{mask}' has shape {tuple(values.shape)}; expected one value per node ({n},).")
            flat.append(values)
        return self.reduce_op(flat)


class BooleanNot(BooleanOperation):
    """Boolean NOT mask."""

    def reduce_op(self, masks: list[torch.Tensor]) -> torch.Tensor:
        assert len(self.masks) == 1, f"The {self.__class__.__name__} can only be aplied to one mask."
        return ~masks[0]


class BooleanAndMask(BooleanOperation):
    """Boolean AND mask."""

    def reduce_op(self, masks: list[torch.Tensor]) -> torch.Tensor:
        out = masks[0]
        for m in masks[1:]:
            out = out & m
        return out


class BooleanOrMask(BooleanOperation):
    """Boolean OR mask."""

    def reduce_op(self, masks: list[torch.Tensor]) -> torch.Tensor:
        out = masks[0]
        for m in masks[1:]:
            out = out | m
        return out
