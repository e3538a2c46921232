"""
The graph hand-off of the reference's mzd/cluster.py (cerebis/bin3C @ 76ad2a9):

    to_graph        cluster.py:278-325     contact map -> weighted undirected graph
    _write_edges    cluster.py:139-151     graph -> 'u v w' edge list consumed by Infomap

to_edges() is the array form of to_graph(): it runs mask -> normalise -> balance -> compress ->
scale on the device and returns one (u, v, w) triple per undirected edge.  to_graph() wraps the
same arrays in the nx.Graph the reference returns; the clustering driver itself (Infomap
subprocess, cluster.py:44-226) is outside the path and consumes either form unchanged.
"""
import logging
import os

import numpy as np

logger = logging.getLogger('mzd.cluster')


def to_edges(contact_map, norm=True, bisto=False, scale=False, min_len=None, min_sig=None, device=False):
    """
    Edge list of the contact graph: u <= v (zero-based gapless ids over the accepted contigs),
    w = value * scl with scl = 1/max over the compressed map incl. its diagonal (Q8).  Self-loops
    are kept, as in the reference (Infomap ignores them).  One value per undirected edge (Q9).

    :param device: return CUDA tensors instead of NumPy arrays
    :return: (u, v, w, scl)
    """
    if not min_len and not min_sig:
        contact_map.set_primary_acceptance_mask()
    else:
        contact_map.set_primary_acceptance_mask(min_len, min_sig, update=True)

    if contact_map._dev.get('processed_map') is None and contact_map.processed_map is None:
        contact_map.prepare_seq_map(norm=norm, bisto=bisto)
    else:
        contact_map.order.set_mask_only(contact_map.get_primary_acceptance_mask())

    if contact_map.is_tipbased():
        # the tensor's 2-D marginal over the accepted sequences (get_subspace(marginalise=True), cluster.py:310),
        # turned into edges by the same device kernels
        import torch
        from . import device as dev
        sub = contact_map.get_subspace(marginalise=True, flatten=False).tocsr()
        keep = dev.to_device(np.ones(sub.shape[0], dtype=np.uint8), torch.uint8)
        res = dev.compress_edges(dev.DeviceCSR.from_scipy(sub, np.float64), keep, want_sub=False, want_edges=True,
                                 scale=scale)
        for k in ('u', 'v', 'w'):
            res[k] = res[k][:res['n_edges']]
    else:
        res = contact_map._subspace_dev(None, want_sub=False, want_edges=True, scale=scale, force=True)
    logger.info('Graph will have {} nodes'.format(contact_map.order.count_accepted()))
    if device:
        return res['u'], res['v'], res['w'], res['scl']
    return (res['u'].cpu().numpy(), res['v'].cpu().numpy(), res['w'].cpu().numpy(), float(res['scl'].cpu()[0]))


def to_graph(contact_map, norm=True, bisto=False, scale=False, extern_ids=False, min_len=None, min_sig=None):
    """
    Convert the seq_map to a undirected Networkx Graph (cluster.py:278-325).

    :param contact_map: an instance of ContactMap to cluster
    :param norm: normalize weights by length
    :param bisto: normalise using bistochasticity
    :param scale: scale weights (max_w = 1)
    :param extern_ids: use the original external sequence identifiers for node ids
    :param min_len: override minimum sequence length, otherwise use instance's setting)
    :param min_sig: override minimum off-diagonal signal (in raw counts), otherwise use instance's setting)
    :return: graph of contigs
    """
    import networkx as nx
    u, v, w, _ = to_edges(contact_map, norm=norm, bisto=bisto, scale=scale, min_len=min_len, min_sig=min_sig)
    logger.debug('Building graph from edges')
    g = nx.Graph(name='contact_graph')
    if extern_ids:
        names = np.array([contact_map.seq_info[i].name for i in contact_map.order.accepted()], dtype=object)
        g.add_weighted_edges_from(zip(names[u].tolist(), names[v].tolist(), w.tolist()))
    else:
        g.add_weighted_edges_from(zip(u.tolist(), v.tolist(), w.tolist()))
    logger.info('Finished: {} nodes, {} edges'.format(g.number_of_nodes(), g.number_of_edges()))
    return g


def write_edges(u, v, w, parent_dir, base_name='cm_graph', sep=' ', py2_str=False, threads=0):
    """
    The file nx.write_edgelist(g, path, data=['weight'], delimiter=' ') produces (cluster.py:139-151):
    one 'u v weight' line per undirected edge.  networkx prints the weight with str(): repr(float) on
    Python 3 (the default here); `py2_str=True` gives what the Python 2.7 the reference pins prints
    ('%.12g', '.0' appended to integer-looking values).  Host arrays are written by the native writer of
    libbin3c_io.so (include/bin3c_io.h: b3c_edges_write_fmt), formatted on a pool of threads.  u, v and w may also
    be CUDA tensors, which are formatted on their device and leave it as text (bam_io.write_edges):

        u, v, w, scl = to_edges(cm, norm=True, bisto=True, scale=True, device=True)
        write_edges(u, v, w, out_dir, py2_str=True)

    Either way the file is the same byte for byte.  Returns the path of the file.
    """
    from . import bam_io
    edge_file = os.path.join(parent_dir, '{}.edges'.format(base_name))
    bam_io.write_edges(u, v, w, edge_file, sep=sep,
                       float_style=bam_io.FLOAT_STR12 if py2_str else bam_io.FLOAT_REPR, threads=threads)
    return edge_file
