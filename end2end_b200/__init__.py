"""end2end_b200 -- a B200-native (sm_100a) CTC engine behind the ``pytorch_end2end`` API.

Hot path only: CTC loss forward+backward and greedy CTC decoding, as hand-written CUDA kernels in
``libe2e_ctc.so`` (C ABI in ``include/e2e_ctc.h``).  See DESIGN.md / INTEGRATION.md.
"""
from .decoders.ctc_decoder import AlignmentResults, CTCDecoder, CTCDecoderError, DecoderResults, ErrorCounts, NBestBiasResults, NBestLMResults, NBestResults
from .encoders.text_encoders import CTCEncoder
from .engine import CTCGreedyEngine, CTCLossEngine, GraphedStep
from .functions.forward_backward import ForwardBackwardLossFunction
from .lm import NGramLM, PhraseBias
from .modules.ctc_loss import CTCLoss, ForwardBackwardLossBase, GraphedCTCStep
from .modules.ctc_score import CTCScore
from .modules.mwer_loss import MWERLoss

__all__ = ["CTCLoss", "CTCScore", "MWERLoss", "CTCDecoder", "CTCEncoder", "CTCLossEngine", "CTCGreedyEngine",
           "ForwardBackwardLossFunction", "ForwardBackwardLossBase", "CTCDecoderError", "DecoderResults", "NBestResults", "AlignmentResults",
           "ErrorCounts", "NBestLMResults", "NBestBiasResults", "NGramLM", "PhraseBias",
           "GraphedStep", "GraphedCTCStep"]
__version__ = "0.1.0"
