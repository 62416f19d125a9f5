"""Stand-in for models/lib/base_models.py of the original project: a module of the `models.lib` package that this
repository does not provide. Imports of it must resolve to the checkout's own file."""
