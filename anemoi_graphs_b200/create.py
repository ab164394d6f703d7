"""Graph creator (/root/reference/src/anemoi/graphs/create.py:26-188).

Same recipe schema, same order of operations (node builders, then for every edge set its builders and ONE
attribute registration on the merged edge set by the last builder, :83-90), same ``clean`` /
``post_process`` / ``save`` semantics.  The whole update runs inside one deferred-copy scope: kernels and
device->host copies are enqueued back to back and awaited once.
"""

from __future__ import annotations

import logging
from itertools import chain
from pathlib import Path
from warnings import warn

import torch

from . import device as _device
from .config import DotDict
from .config import instantiate
from .graph import HeteroData

LOGGER = logging.getLogger(__name__)


class GraphCreator:
    """Graph creator."""

    config: DotDict

    def __init__(self, config: str | Path | DotDict | dict):
        if isinstance(config, Path) or isinstance(config, str):
            self.config = DotDict.from_file(config)
        elif isinstance(config, DotDict):
            self.config = config
        else:  # omegaconf DictConfig / plain mapping
            self.config = DotDict(_to_container(config))

        # Support previous version. This will be deprecated in a future release
        edges = []
        for edges_cfg in self.config.get("edges", []):
            if "edge_builder" in edges_cfg:
                warn(
                    "This format will be deprecated. The key 'edge_builder' is renamed to 'edge_builders' and takes a list of edge builders. In addition, the source_mask_attr_name & target_mask_attr_name fields are moved under the each edge builder.",
                    DeprecationWarning,
                    stacklevel=2,
                )

                edge_builder_cfg = edges_cfg.get("edge_builder")
                if edge_builder_cfg is not None:
                    edge_builder_cfg = DotDict(edge_builder_cfg)
                    edge_builder_cfg.source_mask_attr_name = edges_cfg.get("source_mask_attr_name", None)
                    edge_builder_cfg.target_mask_attr_name = edges_cfg.get("target_mask_attr_name", None)
                    edges_cfg["edge_builders"] = [edge_builder_cfg]

            edges.append(edges_cfg)
        self.config.edges = edges
        self._validate()

    # limits of the CUDA path (DESIGN.md section 7): found here, before any kernel runs, instead of mid-build
    MAX_KNN_K = 64
    MAX_X_HOPS = 8
    EARLY_ROW_MIN_TARGETS = 1 << 18  # smaller target sets: the a-priori target row is not worth a separate copy

    def _validate(self) -> None:
        """Resolve every ``_target_`` of the recipe (an unknown or unbuilt class - the ICON builders,
        ``PlanarAreaWeights`` - raises ImportError now), check the grid names of ``ReducedGaussianGridNodes`` and the
        limits of the kernels."""
        from .config import resolve_target

        def walk(cfg):
            if isinstance(cfg, dict):
                if "_target_" in cfg:
                    resolve_target(cfg["_target_"])
                for v in cfg.values():
                    walk(v)
            elif isinstance(cfg, (list, tuple)):
                for v in cfg:
                    walk(v)

        walk(self.config.get("nodes", {}))
        walk(self.config.get("edges", []))
        walk(self.config.get("post_processors", []))
        from .edges.builder import check_scale_levels
        from .edges.builder import scale_levels
        from .nodes.builders.from_reduced_gaussian import octahedral_number

        for nodes_cfg in self.config.get("nodes", {}).values():
            node_builder = nodes_cfg.get("node_builder", {})
            if str(node_builder.get("_target_", "")).rsplit(".", 1)[-1] == "ReducedGaussianGridNodes":
                octahedral_number(node_builder.get("grid"))
        for edges_cfg in self.config.get("edges", []):
            for b in edges_cfg.get("edge_builders", []):
                target = str(b.get("_target_", ""))
                name = target.rsplit(".", 1)[-1]
                k, hops = b.get("num_nearest_neighbours"), b.get("x_hops")
                if name in ("KNNEdges", "ReversedKNNEdges") and isinstance(k, int) and k > self.MAX_KNN_K:
                    raise NotImplementedError(f"{name}: num_nearest_neighbours = {k} > {self.MAX_KNN_K} is not built")
                if name == "MultiScaleEdges" and isinstance(hops, int) and hops > self.MAX_X_HOPS:
                    raise NotImplementedError(f"MultiScaleEdges: x_hops = {hops} > {self.MAX_X_HOPS} is not built")
                if name == "MultiScaleEdges" and b.get("scale_resolutions") is not None:
                    levels = scale_levels(b.get("scale_resolutions"))
                    check_scale_levels(levels, self._finest_level(edges_cfg.get("source_name")))

    def _finest_level(self, nodes_name) -> int | None:
        """The finest refinement level of a node set the recipe builds (``resolution`` / ``lam_resolution`` of its node
        builder), or None when the recipe does not say."""
        node_builder = self.config.get("nodes", {}).get(nodes_name, {}).get("node_builder", {})
        res = node_builder.get("lam_resolution", node_builder.get("resolution"))
        if isinstance(res, int) and not isinstance(res, bool):
            return res
        if isinstance(res, (list, tuple)) and res and all(isinstance(r, int) for r in res):
            return max(res)
        return None

    def update_graph(self, graph):
        """Instantiate the node and edge builders of the recipe and apply them to the graph (create.py:62-92)."""
        with _device.deferred():
            # host coordinates of node sets the graph arrives with start their way to the device before anything else
            named = {n for e in self.config.get("edges", {}) for n in (e.get("source_name"), e.get("target_name"))}
            for name in named:
                if name in graph.node_types and name not in self.config.get("nodes", {}):
                    _device.prefetch_coordinates(graph[name])
            for nodes_name, nodes_cfg in self.config.get("nodes", {}).items():
                node_builder = instantiate(nodes_cfg.node_builder, name=nodes_name)
                _device.flush_for(node_builder)  # a foreign (reference-style) plugin reads complete host tensors
                graph = node_builder.update_graph(graph, attrs_config=nodes_cfg.get("attributes", {}))

            self._emit_known_rows(graph)
            for edges_cfg in self.config.get("edges", {}):
                for edge_builder_cfg in edges_cfg.edge_builders:
                    edge_builder = instantiate(
                        edge_builder_cfg, source_name=edges_cfg.source_name, target_name=edges_cfg.target_name
                    )
                    _device.flush_for(edge_builder)
                    graph = edge_builder.update_graph(graph, attrs_config=None)

                _device.flush_for(edge_builder)
                graph = edge_builder.register_attributes(graph, edges_cfg.get("attributes", {}))

        return graph

    def _emit_known_rows(self, graph) -> None:
        """Host-resident graphs: the target row of an edge set built by ONE unmasked KNNEdges over a node set the graph
        arrived with is known before any search (``device.emit_regular_target_row``) and starts its way to the host now,
        behind the node builders' own copies."""
        from .config import resolve_target
        from .edges import KNNEdges

        if not torch.cuda.is_available() or _device.is_resident() or _device.sharded_output():
            return
        for edges_cfg in self.config.get("edges", {}):
            builders = edges_cfg.get("edge_builders", [])
            if len(builders) != 1:
                continue
            b = builders[0]
            src, dst, k = edges_cfg.get("source_name"), edges_cfg.get("target_name"), b.get("num_nearest_neighbours")
            try:
                ours = resolve_target(str(b.get("_target_", ""))) is KNNEdges
            except Exception:
                ours = False
            if not ours or not isinstance(k, int) or k <= 0 or k > self.MAX_KNN_K:
                continue
            if b.get("source_mask_attr_name") is not None or b.get("target_mask_attr_name") is not None:
                continue
            if dst not in graph.node_types or dst in self.config.get("nodes", {}) or (src, "to", dst) in graph.edge_types:
                continue
            x = graph[dst].get("x", None)
            if isinstance(x, torch.Tensor) and not x.is_cuda and x.dim() == 2 and int(x.shape[0]) >= self.EARLY_ROW_MIN_TARGETS:
                _device.emit_regular_target_row(int(x.shape[0]), k)

    def clean(self, graph):
        """Remove private attributes used during creation from the graph (create.py:94-114)."""
        LOGGER.info("Cleaning graph.")
        for type_name in chain(graph.node_types, graph.edge_types):
            attr_names_to_remove = [attr_name for attr_name in graph[type_name] if attr_name.startswith("_")]
            for attr_name in attr_names_to_remove:
                del graph[type_name][attr_name]
                LOGGER.info(f"{attr_name} deleted from graph.")

        return graph

    def post_process(self, graph):
        """Apply the configured post-processors, in order (create.py:116-140)."""
        for processor in self.config.get("post_processors", []):
            processor = instantiate(processor)
            _device.flush_for(processor)
            graph = processor.update_graph(graph)

        return graph

    def save(self, graph, save_path: Path, overwrite: bool = False) -> None:
        """Save the generated graph to the output path (create.py:142-161)."""
        save_path = Path(save_path)

        if not save_path.exists() or overwrite:
            save_path.parent.mkdir(parents=True, exist_ok=True)
            torch.save(graph, save_path)
            LOGGER.info(f"Graph saved at {save_path}.")
        else:
            LOGGER.info("Graph already exists. Use overwrite=True to overwrite.")

    def create(self, save_path: Path | None = None, overwrite: bool = False):
        """Create the graph and save it to the output path (create.py:163-188)."""
        graph = HeteroData()
        graph = self.update_graph(graph)
        graph = self.clean(graph)
        graph = self.post_process(graph)

        if save_path is None:
            LOGGER.warning("No output path specified. The graph will not be saved.")
        else:
            self.save(graph, save_path, overwrite)

        return graph


def _to_container(config):
    try:  # pragma: no cover - omegaconf is not in this image
        from omegaconf import DictConfig, OmegaConf

        if isinstance(config, DictConfig):
            return OmegaConf.to_container(config, resolve=True)
    except ImportError:
        pass
    return dict(config)
