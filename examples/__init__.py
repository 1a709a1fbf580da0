"""User environments written for this library; each module registers its environments with envs.register."""
