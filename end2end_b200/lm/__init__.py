"""Word language models for the GPU prefix beam search."""
from .ngram import NGramLM

__all__ = ["NGramLM"]
