"""Word language models and phrase biasing for the GPU prefix beam search."""
from .bias import PhraseBias
from .ngram import NGramLM

__all__ = ["NGramLM", "PhraseBias"]
