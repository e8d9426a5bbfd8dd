"""idelucs_b200 — B200-native (sm_100a CUDA behind a C ABI) implementation of the iDeLUCS
featurisation / mimic / IIC-loss hot path, with the reference's Python call signatures.

Reference surface mirrored (idelucs/__init__.py:3-8): ``check_sequence``, ``SummaryFasta``, ``reverse_complement``,
``kmer_rev_comp``, ``kmersFasta``, ``cgrFasta``, ``cluster_acc``, ``compute_results``, ``SequenceDataset``, ``kmer_counts``,
``cgr``, ``IID_model``, ``IID_loss``, ``info_nce_loss``, ``iDeLUCS_cluster`` (``PlotPolygon`` / ``define_ToolTips`` are GUI / plot
helpers and out of scope).
Submodules keep the reference's names: ``kmers``, ``utils``, ``LossFunctions``, ``models``,
``cluster``.  ``hdbscan_device`` is sklearn's HDBSCAN and ``silhouette_samples_device`` /
``silhouette_score_device`` are sklearn's silhouette metrics, each with its all-pairs work on the GPU.  Nothing here falls back to a CPU implementation.
"""
__version__ = (0, 1, 0)

__all__ = ["kmers", "utils", "LossFunctions", "models", "cluster", "seqset", "featurise", "hdbscan", "metrics"]


def __getattr__(name):  # lazy: importing the package must not require torch.cuda to be usable
    import importlib
    lazy = {
        "kmer_counts": ("kmers", "kmer_counts"),
        "cgr": ("kmers", "cgr"),
        "reverse_complement": ("utils", "reverse_complement"),
        "kmer_rev_comp": ("utils", "kmer_rev_comp"),
        "cgrFasta": ("utils", "cgrFasta"),
        "cluster_acc": ("utils", "cluster_acc"),
        "compute_results": ("utils", "compute_results"),
        "label_features": ("utils", "label_features"),
        "check_sequence": ("utils", "check_sequence"),
        "kmersFasta": ("utils", "kmersFasta"),
        "AugmentFasta": ("utils", "AugmentFasta"),
        "SequenceDataset": ("utils", "SequenceDataset"),
        "SummaryFasta": ("utils", "SummaryFasta"),
        "IID_loss": ("LossFunctions", "IID_loss"),
        "info_nce_loss": ("LossFunctions", "info_nce_loss"),
        "IID_model": ("models", "IID_model"),
        "iDeLUCS_cluster": ("cluster", "iDeLUCS_cluster"),
        "hdbscan_device": ("hdbscan", "hdbscan_device"),
        "silhouette_samples_device": ("metrics", "silhouette_samples_device"),
        "silhouette_score_device": ("metrics", "silhouette_score_device"),
    }
    if name in lazy:
        mod, attr = lazy[name]
        return getattr(importlib.import_module("idelucs_b200." + mod), attr)
    if name in __all__:
        return importlib.import_module("idelucs_b200." + name)
    raise AttributeError(name)
