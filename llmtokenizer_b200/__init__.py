"""B200-native BPE merge-loop engine behind neofytr/LLMTokenizer's C API (see DESIGN.md)."""
from .bpe import (BpeCudaError, Context, compress, decode, decode_batch, dump_pairs, encode, encode_batch, encode_file, get_file, nccl_unique_id, print_text,
                  train_file,
                  read_pairs, train)

__all__ = ["BpeCudaError", "Context", "compress", "decode", "decode_batch", "dump_pairs", "encode", "encode_batch", "encode_file", "train_file", "get_file", "nccl_unique_id", "print_text",
           "read_pairs", "train"]
