// oi_tokenize.cuh — the tokenizer's byte classes (docs/SPEC.md §6), shared by the lexicon scorer (lexicon.cu) and the
// text index builder (text_index.cu) so that both kernels cut the same tokens.
//
// Unicode-lowercase, split on every char that is not ASCII alphanumeric.  On UTF-8 bytes: ASCII letters/digits are
// token bytes (A-Z lowered), every other byte is a separator, except U+212A KELVIN SIGN (E2 84 AA -> 'k', its two
// continuation bytes are transparent) and U+0130 (C4 B0 -> 'i' followed by a separator).
#pragma once
#include <stdint.h>

enum { CLS_SEP = 0, CLS_SKIP = -1, CLS_I_THEN_SEP = -2 };  // > 0: a token byte (the lowered char)

// an ASCII byte that is a token byte ([0-9A-Za-z])
__device__ __forceinline__ bool oi_ascii_token_byte(uint32_t b) { return ((b | 0x20u) - 'a') < 26u || (b - '0') < 10u; }

// class of byte position i of text[0..len): token char (> 0), separator, transparent, or the
// 'i' of U+0130 (a token char that also ends the token)
__device__ __forceinline__ int classify(const uint8_t *t, long long i, long long len) {
  const uint8_t b = t[i];
  if (b < 0x80) {
    if (b >= 'A' && b <= 'Z') return b + 32;
    if ((b >= 'a' && b <= 'z') || (b >= '0' && b <= '9')) return b;
    return CLS_SEP;
  }
  if (b == 0xE2 && i + 2 < len && t[i + 1] == 0x84 && t[i + 2] == 0xAA) return 'k';
  if (b == 0x84 && i >= 1 && i + 1 < len && t[i - 1] == 0xE2 && t[i + 1] == 0xAA) return CLS_SKIP;
  if (b == 0xAA && i >= 2 && t[i - 2] == 0xE2 && t[i - 1] == 0x84) return CLS_SKIP;
  if (b == 0xC4 && i + 1 < len && t[i + 1] == 0xB0) return CLS_I_THEN_SEP;
  return CLS_SEP;
}
