"""B200-native GRUDecoder + CTC hot path of EdwardoSunny/Neural-Speech-Decoder.

Public surface (mirrors the reference's, SURVEY.md section 8b):
    GRUDecoder            src/neural_decoder/model.py:7-123
    NeuralTransformerCTCModel   src/neural_decoder/transformer_ctc.py:333-501 (+ conformer_loss / FusedAdamW: trainer:137-162, 206-260)
    CTCLoss               torch.nn.CTCLoss as used at neural_decoder_trainer.py:139-141
    greedy_decode / phoneme_error_rate      trainer:313-333
    CtcBeamSearch / ctc_beam_search         prefix beam search with a phoneme-bigram prior, N-best (no counterpart)
    ctc_forced_align / frames_to_bins       per-phoneme timing and scores of the true transcript (no counterpart)
    StreamingDecoder / StreamingSessions    stateful streaming inference, lockstep batch / independent sessions (no counterpart)
    train_step / eval_batch / align_batch   trainer:181-260 / 286-333 (hot-loop lines only) / eval_batch's alignment twin
    input_attribution                       saliency / integrated gradients of each utterance's CTC NLL w.r.t. the input (no counterpart)
    input_noise                             trainer:194-201 (white noise + constant offset; also fused into the front end)
All compute is in ``libnsd_b200.so`` (include/nsd_b200.h); there is no CPU or PyTorch fallback.
"""
from ._lib import NsdError, lib  # noqa: F401
from .model import GRUDecoder, set_default_precision  # noqa: F401
from .ctc import (CTCLoss, ctc_loss_from_logits, greedy_decode, decoded_to_lists, edit_distances,  # noqa: F401
                  phoneme_error_rate, out_lens, CtcBeamSearch, ctc_beam_search, CtcAlignment, ctc_forced_align, frames_to_bins)
from .trainer import train_step, eval_batch, align_batch, input_attribution, make_optimizer, LossReader  # noqa: F401
from .ops import input_noise  # noqa: F401   trainer:194-201 as one kernel
from .streaming import StreamingDecoder  # noqa: F401   stateful incremental inference (no counterpart in the reference)
from .streaming import StreamingSessions  # noqa: F401   independent per-slot streaming sessions (no counterpart in the reference)
from .conformer import (NeuralTransformerCTCModel, conformer_loss, conformer_train_step, FusedAdamW, lr_lambda, GraphedConformerStep)  # noqa: F401   transformer_ctc.py:333-501
from .data import BatchPrefetcher  # noqa: F401   trainer:185-191 (H2D copies) overlapped with the previous step

__version__ = "0.1.0"
