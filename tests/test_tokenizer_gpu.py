"""The tokenizer parity tests again under the `gpu` marker, so a `-m gpu` run includes them (they need no GPU; that selection
would otherwise deselect the whole tokenizer suite). The real-vocabulary cases (the known-answer vector of
src/token/clip.rs:232-249 among them) run on the stored vocabulary subset, like everything else in test_tokenizer.py."""
import pytest

import test_tokenizer as T

pytestmark = pytest.mark.gpu
mini = T.mini
real = T.real

test_mini_vocab_vectors = T.test_mini_vocab_vectors
test_case_fold_closure_of_letter_class = T.test_case_fold_closure_of_letter_class
test_fuzz_cxx_equals_oracle_mini = T.test_fuzz_cxx_equals_oracle_mini
test_truncation_drops_end_of_text = T.test_truncation_drops_end_of_text
test_errors_are_reported_not_thrown_across_the_abi = T.test_errors_are_reported_not_thrown_across_the_abi
test_invalid_utf8_is_replaced_like_from_utf8_lossy = T.test_invalid_utf8_is_replaced_like_from_utf8_lossy
test_reference_known_answer_pins_the_oracle = T.test_reference_known_answer_pins_the_oracle
test_reference_known_answer_cxx = T.test_reference_known_answer_cxx
test_fuzz_cxx_equals_oracle_real = T.test_fuzz_cxx_equals_oracle_real
