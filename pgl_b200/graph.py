"""Graph / DistGPUGraph: PGL's graph container and send/recv dispatch (mirror of reference
pgl/graph.py) with torch CUDA tensors as the device container and libpglb's sm_100a kernels
behind every tensor-mode operation.

What differs from the reference by design (DESIGN.md):
 * the fused ``send_recv`` family runs node-parallel over the *cached* dst-keyed CSR instead
   of re-slicing ``edges[:, 0] / edges[:, 1]`` and scatter-adding with atomics on every call
   (reference graph.py:859-860);
 * tensor-mode CSR construction is stable (device radix sort), so ``sorted_edges`` is the same
   in numpy and tensor mode;
 * tensor mode means CUDA: there is no CPU tensor path.
"""
import json
import os
import warnings

import numpy as np
import torch

from . import ops
from .message import Message
from .utils import op
from .utils.edge_index import EdgeIndex, sorted_successor_csr
from .utils.helper import (check_is_tensor, generate_segment_id_from_index, maybe_num_nodes,
                           to_tensor)

__all__ = ["Graph", "DistGPUGraph"]


def _as_int(n):
    if isinstance(n, torch.Tensor):
        return int(n.item())
    return int(n)


class Graph(object):
    """Homogeneous graph (reference pgl/graph.py:38-188).

    Args:
        edges: list of (u, v) tuples, [E, 2] numpy.ndarray or torch.Tensor (int64).
        num_nodes: optional node count (default max(edges) + 1).
        node_feat / edge_feat: optional dicts name -> array / tensor.

    If any argument is a tensor the whole graph is in tensor mode (CUDA); otherwise numpy mode.
    ``send`` / ``recv`` / ``send_recv`` need tensor mode (``Graph.tensor()``).
    """

    def __init__(self, edges, num_nodes=None, node_feat=None, edge_feat=None, **kwargs):
        self._node_feat = node_feat if node_feat is not None else {}
        self._edge_feat = edge_feat if edge_feat is not None else {}

        if not check_is_tensor(edges):
            if isinstance(edges, np.ndarray):
                if edges.dtype != "int64":
                    edges = edges.astype("int64")
            else:
                edges = np.array(edges, dtype="int64")
            edges = edges.reshape(-1, 2)
        self._edges = edges

        self._num_nodes = maybe_num_nodes(self._edges) if num_nodes is None else num_nodes
        self._adj_src_index = kwargs.get("adj_src_index", None)
        self._adj_dst_index = kwargs.get("adj_dst_index", None)

        if check_is_tensor(self._num_nodes, self._edges, *list(self._node_feat.values()),
                           *list(self._edge_feat.values())):
            self._is_tensor = True
        elif self._adj_src_index is not None and self._adj_src_index.is_tensor():
            self._is_tensor = True
        elif self._adj_dst_index is not None and self._adj_dst_index.is_tensor():
            self._is_tensor = True
        else:
            self._is_tensor = False

        if self._is_tensor:
            self._n = _as_int(self._num_nodes)
            self._num_nodes = to_tensor(np.int64(self._n)) if not check_is_tensor(self._num_nodes) \
                else to_tensor(self._num_nodes)
            self._edges = to_tensor(self._edges)
            if self._edges.dtype != torch.int64:
                self._edges = self._edges.to(torch.int64)
            self._edges = self._edges.reshape(-1, 2).contiguous()
            for key in self._node_feat:
                self._node_feat[key] = to_tensor(self._node_feat[key])
            for key in self._edge_feat:
                self._edge_feat[key] = to_tensor(self._edge_feat[key])
            if self._adj_src_index is not None and not self._adj_src_index.is_tensor():
                self._adj_src_index.tensor(inplace=True)
            if self._adj_dst_index is not None and not self._adj_dst_index.is_tensor():
                self._adj_dst_index.tensor(inplace=True)
        else:
            self._n = int(self._num_nodes)

        self._process_graph_info(**kwargs)
        self._nodes = None

    def __repr__(self):
        repr_dict = {"class": self.__class__.__name__, "num_nodes": int(self._n),
                     "edges_shape": list(self.edges.shape), "node_feat": [], "edge_feat": []}
        for key, value in self.node_feat.items():
            repr_dict["node_feat"].append(
                {"name": key, "shape": list(value.shape), "dtype": str(value.dtype)})
        for key, value in self.edge_feat.items():
            repr_dict["edge_feat"].append(
                {"name": key, "shape": list(value.shape), "dtype": str(value.dtype)})
        return json.dumps(repr_dict, ensure_ascii=False)

    # ------------------------------------------------------------------
    # numpy <-> tensor (reference graph.py:222-353)
    # ------------------------------------------------------------------
    _CONVERT_KEYS = ("_num_nodes", "_edges", "_node_feat", "_edge_feat", "_adj_src_index",
                     "_adj_dst_index", "_num_graph", "_graph_node_index", "_graph_edge_index")

    def is_tensor(self):
        return self._is_tensor

    def _convert(self, value, to_t, inplace):
        if value is None:
            return None
        if isinstance(value, EdgeIndex):
            return value.tensor(inplace=inplace) if to_t else value.numpy(inplace=inplace)
        conv = (lambda v: to_tensor(v)) if to_t else \
            (lambda v: v.cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v))
        if isinstance(value, dict):
            if inplace:
                for k in list(value.keys()):
                    value[k] = conv(value[k])
                return value
            return {k: conv(v) for k, v in value.items()}
        return conv(value)

    def _switch(self, to_t, inplace):
        new = {k: self._convert(self.__dict__.get(k), to_t, inplace) for k in self._CONVERT_KEYS}
        if inplace:
            self.__dict__.update(new)
            self._is_tensor = to_t
            if not to_t:
                self._num_nodes = int(self._n)
                ng = self.__dict__.get("_num_graph")
                if isinstance(ng, np.ndarray):
                    self._num_graph = int(ng.reshape(-1)[0])
            self._nodes = None
            for a in ("_dst_uniq_ind", "_dst_segment_ids", "_src_uniq_ind", "_src_segment_ids", "_succ_csr"):
                self.__dict__.pop(a, None)
            return self
        num_nodes = new["_num_nodes"] if to_t else int(self._n)
        return self.__class__(
            num_nodes=num_nodes, edges=new["_edges"], node_feat=new["_node_feat"],
            edge_feat=new["_edge_feat"], adj_src_index=new["_adj_src_index"],
            adj_dst_index=new["_adj_dst_index"], _num_graph=new["_num_graph"],
            _graph_node_index=new["_graph_node_index"],
            _graph_edge_index=new["_graph_edge_index"])

    def tensor(self, inplace=True, uva=False):
        """Convert to tensor (CUDA) mode; reference graph.py:227-264 (UVA is out of scope)."""
        if self._is_tensor:
            return self
        if uva:
            raise ValueError("uva tensor graph is not supported by pgl_b200")
        return self._switch(True, inplace)

    def numpy(self, inplace=True):
        """Convert to numpy mode; reference graph.py:266-303."""
        if not self._is_tensor:
            return self
        return self._switch(False, inplace)

    # ------------------------------------------------------------------
    # basic information (reference graph.py:359-469)
    # ------------------------------------------------------------------
    @property
    def num_nodes(self):
        return self._num_nodes

    @property
    def num_edges(self):
        return self._edges.shape[0]

    @property
    def nodes(self):
        if self._nodes is None:
            if self.is_tensor():
                self._nodes = torch.arange(self._n, device=self._edges.device)
            else:
                self._nodes = np.arange(self._n)
        return self._nodes

    @property
    def edges(self):
        return self._edges

    def sorted_edges(self, sort_by="src"):
        """(sorted_src, sorted_dst, sorted_eid); reference graph.py:392-413."""
        if sort_by not in ["src", "dst"]:
            raise ValueError("sort_by should be in 'src' or 'dst'.")
        if sort_by == "src":
            src, dst, eid = self.adj_src_index.triples()
        else:
            dst, src, eid = self.adj_dst_index.triples()
        return src, dst, eid

    @property
    def node_feat(self):
        return self._node_feat

    @property
    def edge_feat(self):
        return self._edge_feat

    def indegree(self, nodes=None):
        """reference graph.py:427-448."""
        if nodes is None:
            return self.adj_dst_index.degree
        if self._is_tensor:
            return ops.gather_rows(self.adj_dst_index.degree, to_tensor(nodes))
        return self.adj_dst_index.degree[nodes]

    def outdegree(self, nodes=None):
        """reference graph.py:450-469."""
        if nodes is None:
            return self.adj_src_index.degree
        if self._is_tensor:
            return ops.gather_rows(self.adj_src_index.degree, to_tensor(nodes))
        return self.adj_src_index.degree[nodes]

    def successor(self, nodes=None, return_eids=False):
        """reference graph.py:475-507 (numpy mode only)."""
        if self._is_tensor:
            raise ValueError("You must call Graph.numpy() first. Tensor object don't supprt successor now.")
        if return_eids:
            return self.adj_src_index.view_v(nodes), self.adj_src_index.view_eid(nodes)
        return self.adj_src_index.view_v(nodes)

    def predecessor(self, nodes=None, return_eids=False):
        """reference graph.py:575-607 (numpy mode only)."""
        if self._is_tensor:
            raise ValueError("You must call Graph.numpy() first. Tensor object don't supprt predecessor now.")
        if return_eids:
            return self.adj_dst_index.view_v(nodes), self.adj_dst_index.view_eid(nodes)
        return self.adj_dst_index.view_v(nodes)

    # ------------------------------------------------------------------
    # message passing (reference graph.py:694-969)
    # ------------------------------------------------------------------
    def send(self, message_func, src_feat=None, dst_feat=None, edge_feat=None, node_feat=None):
        """Compute messages on every edge; reference graph.py:694-776.

        message_func(src_feat, dst_feat, edge_feat) receives lazily gathered RowReaders and
        must return a dict of [num_edges, ...] tensors."""
        if not self._is_tensor:
            raise ValueError("You must call Graph.tensor() first")
        if (src_feat is not None or dst_feat is not None) and node_feat is not None:
            raise ValueError("Can not use src/dst feat and node feat at the same time")
        src_feat_temp, dst_feat_temp, edge_feat_temp = {}, {}, {}
        if node_feat is not None:
            assert isinstance(node_feat, dict), "The input node_feat must be a dict"
            src_feat_temp.update(node_feat)
            dst_feat_temp.update(node_feat)
        else:
            if src_feat is not None:
                assert isinstance(src_feat, dict), "The input src_feat must be a dict"
                src_feat_temp.update(src_feat)
            if dst_feat is not None:
                assert isinstance(dst_feat, dict), "The input dst_feat must be a dict"
                dst_feat_temp.update(dst_feat)
        if edge_feat is not None:
            assert isinstance(edge_feat, dict), "The input edge_feat must be a dict"
            edge_feat_temp.update(edge_feat)

        src = self._edges[:, 0]  # strided views: the gather kernel reads them in place
        dst = self._edges[:, 1]
        src_reader = op.RowReader(src_feat_temp, src)
        dst_reader = op.RowReader(dst_feat_temp, dst)
        msg = message_func(src_reader, dst_reader, edge_feat_temp)
        if not isinstance(msg, dict):
            raise TypeError(
                "The outputs of the %s function is expected to be a dict, but got %s"
                % (message_func.__name__, type(msg)))
        return msg

    def recv(self, reduce_func, msg, recv_mode="dst"):
        """Aggregate messages with a user reduce function; reference graph.py:778-832.
        Nodes that receive no message get zeros."""
        if not self._is_tensor:
            raise ValueError("You must call Graph.tensor()")
        if not isinstance(msg, dict):
            raise TypeError("The input of msg should be a dict, but receives a %s" % (type(msg)))
        if not callable(reduce_func):
            raise TypeError("reduce_func should be callable")

        src, dst, eid = self.sorted_edges(sort_by=recv_mode)
        msg = op.RowReader(msg, eid)
        uniq_ind, segment_ids = self.get_segment_ids(src, dst, segment_by=recv_mode)
        bucketed_msg = Message(msg, segment_ids)
        output = reduce_func(bucketed_msg)
        output_dim = output.shape[-1]
        init_output = torch.zeros((self._n, output_dim), dtype=output.dtype, device=output.device)
        if int(uniq_ind.shape[0]) == 0:
            return init_output
        return ops.scatter_rows(init_output, uniq_ind, output)

    def _fwd_csr(self):
        return self.adj_dst_index.csr()

    def _bwd_csr(self):
        return self.adj_src_index.csr()

    def _out_rows(self, feature, out_size):
        if out_size is None:
            return int(feature.shape[0])
        out_size = _as_int(out_size)
        return int(feature.shape[0]) if out_size <= 0 else out_size

    def send_recv(self, feature, reduce_func="sum", out_size=None):
        """Copy-source send + built-in reduce; reference graph.py:834-861
        (paddle.geometric.send_u_recv)."""
        if not self._is_tensor:
            raise ValueError("You must call Graph.tensor()")
        assert reduce_func in ["sum", "mean", "max", "min"], \
            "Only support 'sum', 'mean', 'max', 'min' built-in reduce functions."
        return self._send_u_recv(feature, reduce_func, out_size)

    def send_u_recv(self, feature, reduce_op="sum", out_size=None):
        """reference graph.py:863-887."""
        if not self._is_tensor:
            raise ValueError("You must call Graph.tensor()")
        assert reduce_op in ["sum", "mean", "max", "min"], \
            "Only support 'sum', 'mean', 'max', 'min' built-in reduce functions."
        return self._send_u_recv(feature, reduce_op, out_size)

    def _csr_for_rows(self, n_out):
        """dst-CSR resized to n_out rows (out_size > num_nodes pads empty rows; the reference
        requires out_size >= max(dst)+1)."""
        fwd = self._fwd_csr()
        if n_out == self._n:
            return fwd
        key = ("_csr_rows", n_out)
        cached = self.__dict__.get("_csr_rows_cache", {})
        if key in cached:
            return cached[key]
        indptr = fwd["indptr"]
        if n_out > self._n:
            pad = indptr[-1:].expand(n_out - self._n)
            indptr2 = torch.cat([indptr, pad])
            degree2 = torch.cat([fwd["degree"], torch.zeros(n_out - self._n, dtype=torch.int64,
                                                            device=indptr.device)])
        else:
            if self.adj_dst_index.max_degree and int(fwd["degree"][n_out:].sum().item()) > 0:
                raise ValueError("out_size should be equal with or larger than max(dst) + 1")
            indptr2 = indptr[: n_out + 1].contiguous()
            degree2 = fwd["degree"][:n_out].contiguous()
        out = dict(fwd)
        out["indptr"] = indptr2
        out["degree"] = degree2
        cached[key] = out
        self.__dict__["_csr_rows_cache"] = cached
        return out

    def _send_u_recv(self, feature, reduce_op, out_size, scale_src=None, scale_dst=None):
        ops.require_cuda(feature)
        if int(feature.shape[0]) < self._n:
            raise ValueError("feature has %d rows but the graph has %d nodes" % (int(feature.shape[0]), self._n))
        n_out = self._out_rows(feature, out_size)
        fwd = self._csr_for_rows(n_out)
        bwd = self._bwd_csr if (feature.requires_grad and torch.is_grad_enabled()) else None
        return ops.aggregate_copy(feature, fwd, n_out, reduce_op, bwd=bwd, scale_src=scale_src,
                                  scale_dst=scale_dst)

    def host_aggregator(self, num_rows, dim, chunks=2, depth=2):
        """The cached ``ops.HostAggregator`` of this graph for [num_rows, dim] float32 host matrices
        (``submit`` / ``wait`` pipeline successive calls; see its docstring for the buffer contract)."""
        if not self._is_tensor:
            raise ValueError("You must call Graph.tensor()")
        key = ("_host_agg", int(num_rows), int(dim), int(chunks), int(depth))
        agg = self.__dict__.get("_host_agg_cache", {}).get(key)
        if agg is None:
            agg = ops.HostAggregator(self._fwd_csr(), int(num_rows), self._n, int(dim), self._edges.device,
                                     chunks, depth)
            self.__dict__.setdefault("_host_agg_cache", {})[key] = agg
        return agg

    def send_recv_host(self, feature_host, out_host=None, reduce_func="sum", scale_src=None,
                       scale_dst=None, chunks=2):
        """``send_recv`` for a feature matrix in pinned HOST memory (result in pinned host memory):
        the graph stays resident, the features stream through the GPU in column chunks with upload,
        aggregation and download overlapped (``ops.HostAggregator``).  BLOCKING: when it returns,
        ``out_host`` holds the result and ``feature_host`` may be rewritten.  Not in the reference (its
        tensors are device-resident); this is the host-buffer entry the end-to-end number uses."""
        if not self._is_tensor:
            raise ValueError("You must call Graph.tensor()")
        assert reduce_func in ["sum", "mean", "max", "min"], \
            "Only support 'sum', 'mean', 'max', 'min' built-in reduce functions."
        n, d = int(feature_host.shape[0]), int(feature_host.shape[1])
        agg = self.host_aggregator(n, d, chunks, depth=1)
        if out_host is None:
            out_host = torch.empty((self._n, d), dtype=torch.float32, pin_memory=True)
        return agg(feature_host, out_host, reduce_func, scale_src, scale_dst)

    def send_ue_recv(self, feature, edge_feature, message_op="add", reduce_op="sum",
                     out_size=None):
        """x[src] (op) e, then reduce; reference graph.py:889-937
        (paddle.geometric.send_ue_recv; NumPy broadcasting on the feature dims)."""
        if not self._is_tensor:
            raise ValueError("You must call Graph.tensor()")
        assert message_op in ["add", "sub", "mul", "div"], \
            "Only support 'add', 'sub', 'max', 'min' build-in message functions."
        assert reduce_op in ["sum", "mean", "max", "min"], \
            "Only support 'sum', 'mean', 'max', 'min' built-in reduce functions."
        n_out = self._out_rows(feature, out_size)
        fwd = self._csr_for_rows(n_out)
        return ops.aggregate_ue(feature, edge_feature, fwd, n_out, message_op, reduce_op,
                                bwd=self._bwd_csr, edges=self._edges)

    def send_uv(self, src_feature, dst_feature, message_op="add"):
        """out[e] = x[src[e]] (op) y[dst[e]]; reference graph.py:939-966."""
        if not self._is_tensor:
            raise ValueError("You must call Graph.tensor()")
        assert message_op in ["add", "sub", "mul", "div"], \
            "Only support 'add', 'sub', 'max', 'min' build-in message functions."
        return ops.send_uv(src_feature, dst_feature, self._edges[:, 0], self._edges[:, 1],
                           message_op, src_csr=self._bwd_csr, dst_csr=self._fwd_csr)

    def send_ue(self, feature, edge_feature, message_op="add"):
        """reference graph.py:968-969."""
        raise NotImplementedError

    # ------------------------------------------------------------------
    # batching (reference graph.py:975-1175)
    # ------------------------------------------------------------------
    @classmethod
    def disjoint(cls, graph_list, merged_graph_index=False):
        assert len(graph_list) > 0, \
            "The input graph_list of Graph.disjoint has length %s. It should be greater than 0. " \
            % len(graph_list)
        is_tensor = graph_list[0].is_tensor()
        cat = (lambda xs: torch.cat(xs, 0)) if is_tensor else (lambda xs: np.concatenate(xs, 0))
        counts_n = [g._n for g in graph_list]
        counts_e = [int(g.num_edges) for g in graph_list]
        offs = np.concatenate([[0], np.cumsum(counts_n)])
        edges = cat([g.edges + int(offs[i]) for i, g in enumerate(graph_list)])
        node_feat = {k: cat([g.node_feat[k] for g in graph_list]) for k in graph_list[0].node_feat}
        edge_feat = {k: cat([g.edge_feat[k] for g in graph_list]) for k in graph_list[0].edge_feat}
        num_nodes = int(offs[-1])
        if merged_graph_index:
            num_graph = gni = gei = None
        else:
            gni = np.concatenate([[0], np.cumsum(counts_n)]).astype("int64")
            gei = np.concatenate([[0], np.cumsum(counts_e)]).astype("int64")
            num_graph = len(graph_list)
            if is_tensor:
                gni, gei = to_tensor(gni), to_tensor(gei)
                num_graph = to_tensor(np.array([num_graph], dtype="int64"))
        return cls(num_nodes=to_tensor(np.int64(num_nodes)) if is_tensor else num_nodes,
                   edges=edges, node_feat=node_feat, edge_feat=edge_feat, _num_graph=num_graph,
                   _graph_node_index=gni, _graph_edge_index=gei)

    @staticmethod
    def batch(graph_list):
        return Graph.disjoint(graph_list, merged_graph_index=False)

    @property
    def num_graph(self):
        return self._num_graph

    @property
    def graph_node_id(self):
        return generate_segment_id_from_index(self._graph_node_index)

    @property
    def graph_edge_id(self):
        return generate_segment_id_from_index(self._graph_edge_index)

    def _process_graph_info(self, **kwargs):
        """reference graph.py:1330-1367."""
        self._graph_node_index = kwargs.get("_graph_node_index", None)
        self._graph_edge_index = kwargs.get("_graph_edge_index", None)
        if kwargs.get("_num_graph", None) is not None:
            self._num_graph = kwargs["_num_graph"]
            return
        if self._is_tensor:
            dev = self._edges.device
            self._num_graph = torch.ones(1, dtype=torch.int32, device=dev)
            self._graph_node_index = torch.tensor([0, self._n], dtype=torch.int32, device=dev)
            self._graph_edge_index = torch.tensor([0, int(self.num_edges)], dtype=torch.int32,
                                                  device=dev)
        else:
            self._num_graph = 1
            self._graph_node_index = np.array([0, self._n], dtype="int64")
            self._graph_edge_index = np.array([0, self.num_edges], dtype="int64")

    # ------------------------------------------------------------------
    # persistence: same .npy directory layout as the reference (graph.py:1177-1302)
    # ------------------------------------------------------------------
    def dump(self, path):
        if self._is_tensor:
            self.numpy(inplace=False).dump(path)
            return
        if not os.path.exists(path):
            os.makedirs(path)
        np.save(os.path.join(path, "num_nodes.npy"), self._n)
        np.save(os.path.join(path, "edges.npy"), self._edges)
        np.save(os.path.join(path, "num_graph.npy"), self._num_graph)
        if self._adj_src_index is not None:
            self._adj_src_index.dump(os.path.join(path, "adj_src"))
        if self._adj_dst_index is not None:
            self._adj_dst_index.dump(os.path.join(path, "adj_dst"))
        if self._graph_node_index is not None:
            np.save(os.path.join(path, "graph_node_index.npy"), self._graph_node_index)
        if self._graph_edge_index is not None:
            np.save(os.path.join(path, "graph_edge_index.npy"), self._graph_edge_index)

        def dump_feat(feat_path, feat):
            if len(feat) == 0:
                return
            if not os.path.exists(feat_path):
                os.makedirs(feat_path)
            for key in feat:
                np.save(os.path.join(feat_path, key + ".npy"), feat[key])

        dump_feat(os.path.join(path, "node_feat"), self.node_feat)
        dump_feat(os.path.join(path, "edge_feat"), self.edge_feat)

    @classmethod
    def load(cls, path, mmap_mode="r"):
        num_nodes = np.load(os.path.join(path, "num_nodes.npy"), mmap_mode=mmap_mode)
        edges = np.load(os.path.join(path, "edges.npy"), mmap_mode=mmap_mode)
        num_graph = np.load(os.path.join(path, "num_graph.npy"), mmap_mode=mmap_mode)
        kw = {}
        if os.path.isdir(os.path.join(path, "adj_src")):
            kw["adj_src_index"] = EdgeIndex.load(os.path.join(path, "adj_src"), mmap_mode=mmap_mode)
        if os.path.isdir(os.path.join(path, "adj_dst")):
            kw["adj_dst_index"] = EdgeIndex.load(os.path.join(path, "adj_dst"), mmap_mode=mmap_mode)
        for name in ("graph_node_index", "graph_edge_index"):
            p = os.path.join(path, name + ".npy")
            if os.path.exists(p):
                kw["_" + name] = np.load(p, mmap_mode=mmap_mode)

        def load_feat(feat_path):
            feat = {}
            if os.path.isdir(feat_path):
                for item in os.listdir(feat_path):
                    if item.endswith(".npy"):
                        feat[item[:-4]] = np.load(os.path.join(feat_path, item), mmap_mode=mmap_mode)
            return feat

        return cls(edges=edges, num_nodes=int(num_nodes),
                   node_feat=load_feat(os.path.join(path, "node_feat")),
                   edge_feat=load_feat(os.path.join(path, "edge_feat")),
                   _num_graph=int(num_graph), **kw)

    # ------------------------------------------------------------------
    # cached indices (reference graph.py:1308-1328, 1397-1407)
    # ------------------------------------------------------------------
    @property
    def adj_src_index(self):
        """EdgeIndex keyed by src (u = src, v = dst)."""
        if self._adj_src_index is None:
            self._adj_src_index = EdgeIndex.from_edges(
                u=self._edges[:, 0], v=self._edges[:, 1], num_nodes=self._num_nodes, v_bound=self._n)
        return self._adj_src_index

    def successor_csr(self):
        """(indptr, cols) of the successors with every row in ascending order (cached): what the random walks of
        pgl_b200.sampling read, where "is x a successor of v" is a binary search.  indptr is adj_src_index's."""
        csr = self.__dict__.get("_succ_csr")
        if csr is None:
            csr = self._succ_csr = sorted_successor_csr(self._edges[:, 0], self._edges[:, 1], self._n)
        return csr

    @property
    def adj_dst_index(self):
        """EdgeIndex keyed by dst (u = dst, v = src)."""
        if self._adj_dst_index is None:
            self._adj_dst_index = EdgeIndex.from_edges(
                u=self._edges[:, 1], v=self._edges[:, 0], num_nodes=self._num_nodes, v_bound=self._n)
        return self._adj_dst_index

    def node_batch_iter(self, batch_size, shuffle=True):
        """reference graph.py:1369-1395."""
        if self.is_tensor():
            perm = torch.randperm(self._n, device=self._edges.device) if shuffle \
                else torch.arange(self._n, device=self._edges.device)
        else:
            perm = np.arange(self._n)
            if shuffle:
                np.random.shuffle(perm)
        start = 0
        while start < self._n:
            yield perm[start:start + batch_size]
            start += batch_size

    def get_segment_ids(self, src, dst, segment_by="dst"):
        """(uniq_ind, segment_ids) of the sorted key; reference graph.py:1397-1407.  Derived
        from the cached CSR instead of a sort inside paddle.unique; the compact row pointer of
        the non-empty rows rides along on the tensor for the segment kernels."""
        if segment_by not in ("dst", "src"):
            raise ValueError("segment_by should be in 'src' or 'dst'.")
        attr_u, attr_s = "_%s_uniq_ind" % segment_by, "_%s_segment_ids" % segment_by
        if not hasattr(self, attr_u):
            index = self.adj_dst_index if segment_by == "dst" else self.adj_src_index
            uniq, seg = ops.segment_ids_from_indptr(index._indptr, int(self.num_edges))
            indptr = index._indptr
            compact = torch.cat([indptr.index_select(0, uniq), indptr[-1:]]) if uniq.numel() \
                else torch.zeros(1, dtype=torch.int64, device=indptr.device)
            seg._pglb_indptr = compact
            seg._pglb_max_degree = index.max_degree
            setattr(self, attr_u, uniq)
            setattr(self, attr_s, seg)
        return getattr(self, attr_u), getattr(self, attr_s)


class DistGPUGraph(Graph):
    """Multi-GPU full-batch graph with the REFERENCE's semantics (reference
    pgl/graph.py:1410-1553): edges sharded by ``dst % world == rank``, node features
    replicated, every recv / degree result all-reduce-summed.  Kept as the parity mode; the
    partition + halo-exchange path is ``pgl_b200.distributed.ShardedGraph``.
    """

    def __init__(self, graph):
        warnings.warn("DistGPUGraph is an experimental API for Multi-GPU FullBatch Training.")
        shard_edges, shard_edge_feat = self._shard_edges_by_dst(graph.edges, graph.edge_feat)
        super(DistGPUGraph, self).__init__(num_nodes=graph.num_nodes, edges=shard_edges,
                                           node_feat=graph.node_feat, edge_feat=shard_edge_feat)
        if not self.is_tensor():
            self.tensor(inplace=True)

    def _shard_edges_by_dst(self, edges, edge_feat):
        """reference graph.py:1475-1504."""
        import torch.distributed as dist
        world = dist.get_world_size() if dist.is_initialized() else 1
        rank = dist.get_rank() if dist.is_initialized() else 0
        shard_flag = edges[:, 1]
        mask = (shard_flag % world) == rank
        if isinstance(mask, torch.Tensor):
            eid = torch.nonzero(mask, as_tuple=False).reshape(-1)
            shard_edges = edges.index_select(0, eid)
            shard_edge_feat = {k: v.index_select(0, eid.to(v.device)) for k, v in edge_feat.items()}
        else:
            eid = np.arange(edges.shape[0])[mask]
            shard_edges = edges[eid]
            shard_edge_feat = {k: np.asarray(v)[eid] for k, v in edge_feat.items()}
        return shard_edges, shard_edge_feat

    def numpy(self, inplace=True):
        raise ValueError("DistGPUGraph can't convert into numpy")

    def recv(self, reduce_func, msg, recv_mode="dst"):
        if recv_mode != "dst":
            raise ValueError("Currently DistGPUGraph can only support recv_mode=='dst'")
        output = super(DistGPUGraph, self).recv(msg=msg, reduce_func=reduce_func,
                                                recv_mode=recv_mode)
        return op.all_reduce_sum_with_grad(output)

    def indegree(self, nodes=None):
        return op.all_reduce_sum_with_grad(super(DistGPUGraph, self).indegree(nodes=nodes))

    def outdegree(self, nodes=None):
        return op.all_reduce_sum_with_grad(super(DistGPUGraph, self).outdegree(nodes=nodes))

    def send_recv(self, feature, reduce_func="sum", out_size=None):
        output = super(DistGPUGraph, self).send_recv(feature=feature, reduce_func=reduce_func,
                                                     out_size=out_size)
        return op.all_reduce_sum_with_grad(output)

    def send_u_recv(self, feature, reduce_op="sum", out_size=None):
        output = super(DistGPUGraph, self).send_u_recv(feature=feature, reduce_op=reduce_op,
                                                       out_size=out_size)
        return op.all_reduce_sum_with_grad(output)

    def send_ue_recv(self, feature, edge_feature, message_op="add", reduce_op="sum",
                     out_size=None):
        output = super(DistGPUGraph, self).send_ue_recv(
            feature=feature, edge_feature=edge_feature, message_op=message_op,
            reduce_op=reduce_op, out_size=out_size)
        return op.all_reduce_sum_with_grad(output)
