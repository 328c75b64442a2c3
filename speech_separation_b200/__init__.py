"""speech_separation_b200: B200-native (sm_100a) hot path of teasgen/speech_separation (VAT-SS).

Public surface mirrors the reference's `src.model`, `src.loss` and `src.metrics` entry points for
the DPTN-AV separation forward pass, its PIT SI-SNR loss / metrics, STOI / ESTOI and SI-SDR / SDR / SDRi.  All compute happens in
hand-written CUDA kernels inside libvatss_b200.so (C ABI in include/vatss.h).
"""
from .data import SSDataset, collate_fn, make_dataloader
from .inference import Inferencer, MetricTracker
from .lipreader import Lipreading, extract_embeddings, init_lipreader, make_embeddings
from .longform import LongFormSeparator
from .loss import SiSNRLoss, SiSNRWavLoss, pit_sisnr_all
from .metrics import (SDRiMetric, SDRMetric, SISDRMetric, SISNRiMetric, SISNRMetric, STOIMetric, sdr_all,
                      sisdr_all, stoi_all)
from .model import DPRNNEncDec, DPTNAVWavEncDec, DPTNEncDec, DPTNWavEncDec, OverlapAdd, SplitToFolds

__all__ = [
    "DPTNAVWavEncDec", "DPTNWavEncDec", "DPTNEncDec", "DPRNNEncDec", "SplitToFolds", "OverlapAdd",
    "SiSNRLoss", "SiSNRWavLoss", "SISNRMetric", "SISNRiMetric", "pit_sisnr_all", "Inferencer", "MetricTracker", "SSDataset", "collate_fn", "make_dataloader",
    "Lipreading", "init_lipreader", "extract_embeddings", "make_embeddings", "LongFormSeparator", "STOIMetric",
    "stoi_all", "SISDRMetric", "SDRMetric", "SDRiMetric", "sisdr_all", "sdr_all",
]
