"""deepgate -- B200-native drop-in for the hot path of 959AI994/Multi-Gate-VAE (DG_VAE/deepgate).

Same import surface as the reference package (deepgate/__init__.py:1-10): the four models are
imported under one name, so ``deepgate.Model`` is the XAG model, exactly as upstream.
"""
from . import digae_layer, digae_model, digvae_model
from . import dg_ae_model_aig, dg_ae_model_mig, dg_ae_model_xmg, dg_ae_model_xag
from .dg_ae_model_aig import Model
from .dg_ae_model_mig import Model
from .dg_ae_model_xmg import Model
from .dg_ae_model_xag import Model

from .trainer import Trainer
from .data import OrderedData, DataLoader, CudaPrefetcher, DeferredScalars, collate
from . import parser, parser_func, parser_func_others
from .parser import NpzParser, CircuitDataset, read_npz_file
from .parser_func_others import parse_pyg_mlpgate, circuits_to_batch
from .utils import dag_utils
from .simulate import simulate, simulate_counts, label_circuits, write_npz
from .utils.utils import zero_normalization, AverageMeter
from .__version__ import __version__
