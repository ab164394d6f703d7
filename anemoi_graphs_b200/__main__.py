"""``python -m anemoi_graphs_b200 create recipe.yaml graph.pt [--overwrite]`` - the ``anemoi-graphs create``
and ``describe graph.pt`` entry points (/root/reference/src/anemoi/graphs/commands/create.py:22-56, describe.py:16-30) -
and ``export_to_sparse graph.pt OUT_DIR``, which writes edge sets as scipy ``.npz`` matrices (``export.GraphExporter``):
the command of newer releases as far as is known; the pinned reference does not have it."""

from __future__ import annotations

import argparse
import logging
import sys

from .create import GraphCreator


def main(argv=None) -> int:
    parser = argparse.ArgumentParser(prog="anemoi-graphs")
    sub = parser.add_subparsers(dest="command", required=True)
    create = sub.add_parser("create", help="Create a graph from a recipe.")
    create.add_argument("--overwrite", action="store_true", help="Overwrite existing files. This will delete the target graph if it already exists.")
    create.add_argument("config", help="Configuration yaml file path defining the recipe to create the graph.")
    create.add_argument("save_path", help="Path to store the created graph. File format is torch .pt")
    create.add_argument("--description", action="store_false", help="Show the description of the graph.")
    describe = sub.add_parser("describe", help="Describe a graph.")
    describe.add_argument("graph_file", help="Path to the graph (a .PT file).")
    export = sub.add_parser("export_to_sparse", help="Export edge sets as sparse matrices (scipy .npz files).")
    export.add_argument("graph", help="Path to the graph (a .PT file).")
    export.add_argument("output_path", help="Directory of the <source>_to_<target>.npz files.")
    export.add_argument("--edges-attribute-name", default=None, help="Edge attribute giving the values (default: 1 per edge).")
    export.add_argument(
        "--edges-name", nargs=2, action="append", metavar=("SOURCE", "TARGET"), default=None,
        help="An edge set to export (repeatable; default: every edge set).",
    )  # fmt: skip
    args = parser.parse_args(argv)
    logging.basicConfig(level=logging.INFO, format="%(levelname)s %(name)s: %(message)s")
    if args.command == "describe":
        from .describe import GraphDescriptor

        GraphDescriptor(args.graph_file).describe()
        return 0
    if args.command == "export_to_sparse":
        from .export import GraphExporter

        GraphExporter(args.graph, args.output_path, args.edges_name, args.edges_attribute_name).export()
        return 0
    GraphCreator(config=args.config).create(save_path=args.save_path, overwrite=args.overwrite)
    if args.description:  # commands/create.py:52-55: describe the new graph unless --description is given
        from pathlib import Path

        if Path(args.save_path).exists():
            from .describe import GraphDescriptor

            GraphDescriptor(args.save_path).describe()
    return 0


if __name__ == "__main__":
    sys.exit(main())
