// Host-side dispatch from runtime values to template arguments: a generic lambda receives std::integral_constant
// arguments, so a launch site names its kernel template once and skips combinations that must not exist with `if constexpr`.
#pragma once
#include <type_traits>

// f(std::integral_constant<decltype(V), V>{}) for the V... equal to v; returns false, without calling f, when none is
template <auto... V, class T, class F>
bool with(T v, F&& f) {
  return ((v == V && (f(std::integral_constant<decltype(V), V>{}), true)) || ...);
}

// f(std::integral_constant<decltype(V), V>{}) for every V..., in order
template <auto... V, class F>
void each(F&& f) {
  (f(std::integral_constant<decltype(V), V>{}), ...);
}
