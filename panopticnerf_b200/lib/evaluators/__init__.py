from .evaluator import Evaluator, make_evaluator, summarize_stats

__all__ = ["Evaluator", "make_evaluator", "summarize_stats"]
