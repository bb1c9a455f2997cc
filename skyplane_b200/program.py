"""Gateway-program loader: turns the reference's operator-DAG JSON into wired operators and queues.

Same schema the reference's client builds with ``GatewayProgram.to_dict()`` (skyplane/gateway/gateway_program.py:134-156)
and the daemon consumes in ``create_gateway_operators`` (skyplane/gateway/gateway_daemon.py:126-308)::

    [{"partitions": ["0", ...], "value": [ {"op_type": ..., "handle": ..., "children": [ ... ], <op fields> } ]}]

Wiring rules kept from the reference: a node's handle is ``<op_type>_<handle>``; an operator whose first child
is ``mux_and`` feeds a ``GatewayANDQueue`` (every grandchild sees every chunk), ``mux_or`` children share the
private queue their ``mux_and`` parent gave them, operators without children are terminal, an unknown ``op_type``
raises ``ValueError``.  Built in: the B200 stage's op types (``compress_hash`` between ``read_object_store`` and
``send`` on the source gateway, ``decompress_verify`` before ``write_object_store`` on the destination gateway) and the
reference's three file-only operators (``receive``, ``gen_data``, ``write_local``); the daemon's cloud / socket
operators (object store, sender) are supplied by the caller through ``factories``.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Callable, Dict, List, Optional

from skyplane_b200.chunk_store import ChunkStore
from skyplane_b200.gateway_queue import GatewayANDQueue, GatewayQueue
from skyplane_b200.operators import GatewayCompressHash, GatewayDecompressVerify, GatewayOperator

# factory(op_dict, common_kwargs) -> GatewayOperator ; common_kwargs = handle, region, queues, error plumbing, store
Factory = Callable[[Dict, Dict], GatewayOperator]


def _compress_hash(op: Dict, kw: Dict) -> GatewayOperator:
    return GatewayCompressHash(
        **kw,
        n_processes=op.get("num_gpus", 1),
        use_compression=op.get("compress", True),
        block_linked=op.get("block_linked", False),
        max_batch_chunks=op.get("max_batch_chunks", 64),
        max_batch_bytes=op.get("max_batch_bytes", 512 << 20),
        n_gpus=op.get("num_gpus"),
    )


def _decompress_verify(op: Dict, kw: Dict) -> GatewayOperator:
    return GatewayDecompressVerify(**kw, n_processes=op.get("num_gpus", 1), n_gpus=op.get("num_gpus"))


def _receive(op: Dict, kw: Dict) -> GatewayOperator:
    from skyplane_b200.local_operators import GatewayWaitReceiver

    return GatewayWaitReceiver(**kw, n_processes=1)


def _gen_data(op: Dict, kw: Dict) -> GatewayOperator:
    from skyplane_b200.local_operators import GatewayRandomDataGen

    return GatewayRandomDataGen(**kw, size_mb=op["size_mb"], fill=op.get("fill", "zeros"))


def _write_local(op: Dict, kw: Dict) -> GatewayOperator:
    from skyplane_b200.local_operators import GatewayWriteLocal

    return GatewayWriteLocal(**kw, n_processes=1)


# op types that need neither cloud SDKs nor sockets; read/write_object_store and send come from the caller
BUILTIN_FACTORIES: Dict[str, Factory] = {"compress_hash": _compress_hash, "decompress_verify": _decompress_verify,
                                         "receive": _receive, "gen_data": _gen_data, "write_local": _write_local}
_MUX = ("mux_and", "mux_or")


@dataclass
class OperatorGraph:
    operators: Dict[str, GatewayOperator] = field(default_factory=dict)
    terminal_operators: Dict[str, List[str]] = field(default_factory=dict)  # partition -> handles that end the chain
    num_required_terminal: Dict[str, int] = field(default_factory=dict)  # partition -> completions needed per chunk
    n_processes: int = 0

    def start(self):
        for op in self.operators.values():
            op.start_workers()

    def stop(self):
        for op in self.operators.values():
            op.stop_workers()


def _grandchildren(node: Dict) -> List[Dict]:
    kids = node.get("children", [])
    if kids and kids[0]["op_type"] in _MUX:
        return kids[0].get("children", [])
    return kids


def _queue_after(node: Dict) -> Optional[GatewayQueue]:
    kids = node.get("children", [])
    if not kids:
        return None
    return GatewayANDQueue() if kids[0]["op_type"] == "mux_and" else GatewayQueue()


def build_operator_graph(gateway_program: List[Dict], chunk_store: ChunkStore, region: str, error_event, error_queue,
                         factories: Optional[Dict[str, Factory]] = None) -> OperatorGraph:
    """Instantiate and wire the operators of a gateway program (workers are not started)."""
    known = dict(BUILTIN_FACTORIES)
    known.update(factories or {})
    graph = OperatorGraph()

    def wire(in_queue: GatewayQueue, nodes: List[Dict], partitions: List[str]):
        for node in nodes:
            kind = node["op_type"]
            handle = f"{kind}_{node['handle']}"
            in_queue.register_handle(handle)
            below = _grandchildren(node)
            if kind == "mux_or":
                if not isinstance(in_queue, GatewayANDQueue):
                    raise ValueError(f"{handle}: mux_or must sit under a mux_and")
                wire(in_queue.get_handle_queue(handle), below, partitions)
                continue
            if kind == "mux_and":
                raise ValueError(f"{handle}: mux_and may only appear as the first child of an operator or as the program root")
            out_queue = _queue_after(node)
            if isinstance(out_queue, GatewayANDQueue):  # one completion per branch instead of one
                for part in partitions:
                    graph.num_required_terminal[part] += len(below) - 1
            if out_queue is None:
                for part in partitions:
                    graph.terminal_operators[part].append(handle)
            if kind not in known:
                raise ValueError(f"Unsupported op_type {kind}")
            op = known[kind](node, dict(handle=handle, region=region, input_queue=in_queue, output_queue=out_queue,
                                        error_event=error_event, error_queue=error_queue, chunk_store=chunk_store))
            graph.operators[handle] = op
            graph.n_processes += op.n_processes
            if out_queue is not None:
                wire(out_queue, below, partitions)

    for group in gateway_program:
        partitions = [str(p) for p in group["partitions"]]
        nodes = group["value"]
        if nodes and nodes[0]["op_type"] == "mux_and":
            if len(nodes) != 1:
                raise ValueError("mux_and cannot have siblings")
            root: GatewayQueue = GatewayANDQueue()
            nodes = nodes[0].get("children", [])
            required = len(nodes)
        else:
            root = GatewayQueue()
            required = 1
        for part in partitions:
            graph.num_required_terminal[part] = required
            graph.terminal_operators[part] = []
            chunk_store.add_partition(part, root)
        wire(root, nodes, partitions)
    return graph
