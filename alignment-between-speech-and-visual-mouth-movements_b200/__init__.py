"""B200-native AV sync-scoring hot path of Hu-xiao-max/Alignment-Between-Speech-and-Visual-Mouth-Movements.

Host-side mirror of the reference's Python surface for this path (same names, argument meaning and
error behaviour) over the C-ABI library ``libavsync_b200.so`` (``include/avsync.h``):

    model.LipNet                               <- model.py
    utils.decode_prediction                    <- utils.py
    misalignment_detection_train.{DetectorConfig, shift_audio, compute_audio_stats,
        extract_visual_embeddings, FeatureExtractor, MisalignmentDataset, MisalignmentDetector, run_epoch,
        load_lipnet, save_detector}                  utils.evaluate_model
    misalignment_detection_train.{SyncSweeper, sync_sweep, sweep_score_pairs, audio_stats_sweep_ragged, audio_stats_sweep_windows,
        window_bounds}, utils.{ctc_greedy_decode, ctc_beam_decode, CtcLexicon, ctc_forced_align, CtcAlignment,
        align_words, ctc_grammar_decode, CtcGrammar, CtcGrammarResult, ctc_loss}, model.LipNet.gru_head_train, dataset.{GRID_WORDS, GRID_SLOTS, grid_lexicon,
        grid_grammar, read_grid_align}                                                             (new, batched)
    distributed.{shard_range, sweep_sharded, gather_scores, ddp_detector_step, GraphedDetectorStep}        (new, multi-GPU)

Import as ``avsync_b200`` (the directory name is not a valid identifier; ``avsync_b200.py`` at the
repo root aliases it).
"""
from . import _native
from .model import LipNet
from .utils import (CtcAlignment, CtcGrammar, CtcGrammarResult, CtcLexicon, align_words, ctc_beam_decode,
                    ctc_forced_align, ctc_grammar_decode, ctc_greedy_decode, ctc_loss, decode_batch, decode_metrics,
                    decode_prediction, evaluate_model)
from .misalignment_detection_train import (DetectorConfig, FeatureExtractor, MisalignmentDataset, MisalignmentDetector,
                                           SyncSweeper, run_epoch,
                                           audio_stats_sweep, audio_stats_sweep_ragged, audio_stats_sweep_windows, compute_audio_stats,
                                           extract_visual_embeddings, window_bounds,
                                           load_detector, load_lipnet, save_detector, shift_audio, shift_samples, get_video_fps,
                                           resample_audio, default_audio_loader,
                                           sweep_score, sweep_score_pairs, sync_sweep, visual_stats)
from .dataset import GRID_SLOTS, GRID_WORDS, GridPreprocessor, grid_grammar, grid_lexicon, read_grid_align
from . import distributed

__all__ = ["LipNet", "ctc_greedy_decode", "decode_batch", "decode_prediction", "DetectorConfig", "FeatureExtractor",
           "MisalignmentDataset", "MisalignmentDetector", "SyncSweeper", "run_epoch", "evaluate_model", "decode_metrics", "audio_stats_sweep", "audio_stats_sweep_ragged", "audio_stats_sweep_windows", "window_bounds", "compute_audio_stats",
           "extract_visual_embeddings", "load_detector", "load_lipnet", "save_detector", "shift_audio",
           "shift_samples", "get_video_fps", "resample_audio", "default_audio_loader", "sweep_score", "sweep_score_pairs", "sync_sweep", "visual_stats", "GridPreprocessor", "distributed",
           "CtcLexicon", "ctc_beam_decode", "GRID_WORDS", "grid_lexicon",
           "CtcAlignment", "ctc_forced_align", "align_words", "read_grid_align",
           "CtcGrammar", "CtcGrammarResult", "ctc_grammar_decode", "GRID_SLOTS", "grid_grammar", "ctc_loss"]
