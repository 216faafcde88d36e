"""ms_hgnn - B200-native drop-in for the MS-HGNN forward/backward hot path."""
from .lightning_py.hgnn import COM_HGNN, GRF_HGNN
from .lightning_py.hgnn_c2 import GRF_HGNN_C2
from .lightning_py.hgnn_c2_com import COM_HGNN_C2
from .lightning_py.hgnn_k4 import GRF_HGNN_K4
from .lightning_py.hgnn_k4_com import COM_HGNN_K4
from .lightning_py.hgnn_s4_com import COM_HGNN_S4
from .model_batch import ModelBatch, ModelBatchTrainer

__all__ = ["GRF_HGNN", "COM_HGNN", "GRF_HGNN_K4", "GRF_HGNN_C2", "COM_HGNN_K4", "COM_HGNN_C2", "COM_HGNN_S4", "ModelBatch", "ModelBatchTrainer"]
